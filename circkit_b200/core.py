"""Host-side mirror of the reference's library interface over the C ABI (no compute here).

Reference names kept: ``canonicalize``, ``lmsr``, ``lmsr_index`` (lib/src/canonicalize.rs:5,41,54);
batch calls correspond to the worker / consumer closures of src/canonicalize.rs:21-44 and
src/uniq.rs:33-78.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _native as N


class CircKitError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"circkit_b200 error {code}: {msg}")
        self.code = code


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data


class PackedBatch:
    """What ck_pack2_host leaves for ck_*_submit_packed (include/circkit_b200.h, "packed host input"): the A/C/G/T
    records at 2 bits per base in the dense host layout, normalised lengths, symbol lanes, and the bytes of the byte-lane
    records only.  Keeps the arrays alive for as long as the batch is in flight."""

    def __init__(self, offsets, dense, lens, lane, lane_bytes, lane_offsets, lane_total):
        self.offsets, self.dense, self.lens, self.lane = offsets, dense, lens, lane
        self.lane_bytes, self.lane_offsets, self.lane_total = lane_bytes, lane_offsets, lane_total
        self.n = len(offsets) - 1
        self.total = int(offsets[-1]) if len(offsets) else 0

    def struct(self) -> "N.CkPackedBatch":
        return N.CkPackedBatch(_ptr(self.dense), _ptr(self.offsets), _ptr(self.lens), _ptr(self.lane),
                               _ptr(self.lane_bytes) if self.lane_total else None,
                               _ptr(self.lane_offsets) if self.lane_total else None, self.lane_total, self.n)

    @property
    def h2d_bytes(self) -> int:
        """bytes a submit copies to the device"""
        words = (self.total >> 5) + self.n + 1
        return 8 * words + 8 * (self.n + 1) + 5 * self.n + (self.lane_total + 8 * (self.n + 1) if self.lane_total else 0)


def pack2_host(arena: np.ndarray, offsets: np.ndarray, *, normalize: bool = False, threads: int = 0) -> PackedBatch:
    """ck_pack2_host: the multi-threaded host packer (normalise + classify + 2-bit pack; pure host code)."""
    lib = N.lib()
    arena = np.ascontiguousarray(arena, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    n = len(offsets) - 1
    total = int(offsets[-1]) if n >= 0 and len(offsets) else 0
    dense = np.zeros(int(lib.ck_pack2_words(total, max(n, 0))), dtype=np.uint64)
    lens = np.zeros(max(n, 1), dtype=np.uint32)
    lane = np.zeros(max(n, 1), dtype=np.uint8)
    lane_bytes = np.zeros(max(total, 1), dtype=np.uint8)
    lane_offsets = np.zeros(max(n, 0) + 1, dtype=np.uint64)
    lane_total = C.c_uint64(0)
    rc = lib.ck_pack2_host(_ptr(arena), _ptr(offsets), max(n, 0), N.CK_F_NORMALIZE if normalize else 0, threads, _ptr(dense),
                           _ptr(lens), _ptr(lane), _ptr(lane_bytes), total, _ptr(lane_offsets), C.byref(lane_total))
    if rc != N.CK_OK:
        raise CircKitError(rc, "ck_pack2_host: bad batch (offsets not monotonic, record longer than 2^30, or null pointers)")
    return PackedBatch(offsets, dense, lens[:max(n, 0)], lane[:max(n, 0)], lane_bytes, lane_offsets, int(lane_total.value))


class Context:
    """One ``ck_ctx``: a device, two in-flight batch slots, the uniq first-occurrence table."""

    def __init__(self, device: int = 0, max_batch_bytes: int = 64 << 20, max_batch_records: int = 1 << 20,
                 table_capacity: int = 0):
        self._lib = N.lib()
        self._h = C.c_void_p()
        cfg = N.CkConfig(device, max_batch_bytes, max_batch_records, table_capacity)
        rc = self._lib.ck_init(C.byref(cfg), C.byref(self._h))
        if rc != N.CK_OK:
            raise CircKitError(rc, (self._lib.ck_last_error(None) or b"").decode())
        self.device = device
        self.max_batch_bytes = max_batch_bytes
        self.max_batch_records = max_batch_records
        self._text_batch = {}           # slot -> (records, text bytes) of its text batch in flight
        self._deflate_batch = {}        # slot -> (input bytes, input, dict) of its deflate call in flight
        self._bzip2_batch = {}          # slot -> input bytes of its bzip2 call in flight

    # -- plumbing
    @property
    def handle(self):
        return self._h

    def _check(self, rc: int):
        if rc != N.CK_OK:
            raise CircKitError(rc, (self._lib.ck_last_error(self._h) or b"").decode())

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.ck_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def launch_count(self) -> int:
        return int(self._lib.ck_launch_count(self._h))

    # -- library drop-ins (library semantics: bytes as they are)
    def lmsr_index(self, s: bytes) -> int:
        out = C.c_size_t(0)
        self._check(self._lib.ck_lmsr_index(self._h, s, len(s), C.byref(out)))
        return out.value

    def lmsr(self, s: bytes) -> bytes:
        out = C.create_string_buffer(max(len(s), 1))
        self._check(self._lib.ck_lmsr(self._h, s, len(s), out))
        return out.raw[: len(s)]

    def canonicalize(self, s: bytes) -> bytes:
        out = C.create_string_buffer(max(len(s), 1))
        self._check(self._lib.ck_canonicalize(self._h, s, len(s), out))
        return out.raw[: len(s)]

    def lmsr_index_batch(self, arena: np.ndarray, offsets: np.ndarray) -> np.ndarray:
        arena = np.ascontiguousarray(arena, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = len(offsets) - 1
        out = np.zeros(max(n, 1), dtype=np.uint32)
        self._check(self._lib.ck_lmsr_index_batch(self._h, _ptr(arena), _ptr(offsets), n, _ptr(out)))
        return out[:n]

    # -- batch API (host buffers)
    def out_arena_bytes(self, total: int, n: int) -> int:
        """Size of the CK_F_ALIGNED_OUT output arena (record i at 32 * ((offsets[i] >> 5) + i))."""
        return int(self._lib.ck_out_arena_bytes(total, n))

    @staticmethod
    def aligned_starts(offsets: np.ndarray) -> np.ndarray:
        """Byte position of every record in the aligned output arena."""
        off = np.asarray(offsets[:-1], dtype=np.uint64)
        return 32 * ((off >> np.uint64(5)) + np.arange(len(off), dtype=np.uint64))

    def canon_submit(self, slot: int, arena: np.ndarray, offsets: np.ndarray, *, normalize: bool, no_bytes=False,
                     aligned=False):
        flags = ((N.CK_F_NORMALIZE if normalize else 0) | (N.CK_F_NO_BYTES if no_bytes else 0)
                 | (N.CK_F_ALIGNED_OUT if aligned else 0))
        self._check(self._lib.ck_canon_submit(self._h, slot, _ptr(arena), _ptr(offsets), len(offsets) - 1, flags))

    def canon_wait(self, slot: int, n: int, total: int, *, want_bytes=True, aligned=False):
        nbytes = self.out_arena_bytes(total, n) if aligned else total
        out = np.zeros(max(nbytes, 1), dtype=np.uint8) if want_bytes else None
        lens = np.zeros(max(n, 1), dtype=np.uint32)
        start = np.zeros(max(n, 1), dtype=np.uint32)
        strand = np.zeros(max(n, 1), dtype=np.uint8)
        h = np.zeros(max(n, 1), dtype=np.uint64)
        self._check(self._lib.ck_canon_wait(self._h, slot, _ptr(out), _ptr(lens), _ptr(start), _ptr(strand), _ptr(h)))
        return dict(out=None if out is None else out[:nbytes], lens=lens[:n], start=start[:n], strand=strand[:n], hash=h[:n])

    def canonicalize_batch(self, arena: np.ndarray, offsets: np.ndarray, *, normalize: bool = False, want_bytes=True,
                           aligned=False):
        """Worker closure over a batch (src/canonicalize.rs:21-30): returns dict(out, lens, start, strand, hash).
        aligned=True: `out` is the 32-byte-aligned arena (record i at aligned_starts(offsets)[i])."""
        arena = np.ascontiguousarray(arena, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        self.canon_submit(0, arena, offsets, normalize=normalize, no_bytes=not want_bytes, aligned=aligned)
        return self.canon_wait(0, len(offsets) - 1, int(offsets[-1]) if len(offsets) else 0, want_bytes=want_bytes,
                               aligned=aligned)

    # -- batch API, packed host input (2 bits per base over PCIe)
    def canon_submit_packed(self, slot: int, pb: PackedBatch, *, no_bytes=False, aligned=False):
        flags = (N.CK_F_NO_BYTES if no_bytes else 0) | (N.CK_F_ALIGNED_OUT if aligned else 0)
        st = pb.struct()
        self._check(self._lib.ck_canon_submit_packed(self._h, slot, C.byref(st), flags))

    def uniq_submit_packed(self, slot: int, pb: PackedBatch, base_index: int, *, no_bytes=False, aligned=False, survivors=False):
        flags = ((N.CK_F_NO_BYTES if no_bytes else 0) | (N.CK_F_ALIGNED_OUT if aligned else 0)
                 | (N.CK_F_SURVIVORS if survivors else 0))
        st = pb.struct()
        self._check(self._lib.ck_uniq_submit_packed(self._h, slot, C.byref(st), flags, base_index))

    def canonicalize_batch_packed(self, arena: np.ndarray, offsets: np.ndarray, *, normalize: bool = False, want_bytes=True,
                                  aligned=False, threads: int = 0):
        """canonicalize_batch through the packed host path: ck_pack2_host, then ck_canon_submit_packed / ck_canon_wait."""
        pb = pack2_host(arena, offsets, normalize=normalize, threads=threads)
        self.canon_submit_packed(0, pb, no_bytes=not want_bytes, aligned=aligned)
        return self.canon_wait(0, pb.n, pb.total, want_bytes=want_bytes, aligned=aligned)

    def uniq_batch_packed(self, arena: np.ndarray, offsets: np.ndarray, base_index: int = 0, *, normalize: bool = False,
                          want_bytes=True, aligned=False, threads: int = 0):
        pb = pack2_host(arena, offsets, normalize=normalize, threads=threads)
        self.uniq_submit_packed(0, pb, base_index, no_bytes=not want_bytes, aligned=aligned)
        return self.uniq_wait(0, pb.n, pb.total, want_bytes=want_bytes, aligned=aligned)

    def uniq_submit(self, slot: int, arena: np.ndarray, offsets: np.ndarray, base_index: int, *, normalize: bool,
                    no_bytes=False, aligned=False, survivors=False):
        flags = ((N.CK_F_NORMALIZE if normalize else 0) | (N.CK_F_NO_BYTES if no_bytes else 0)
                 | (N.CK_F_ALIGNED_OUT if aligned else 0) | (N.CK_F_SURVIVORS if survivors else 0))
        self._check(self._lib.ck_uniq_submit(self._h, slot, _ptr(arena), _ptr(offsets), len(offsets) - 1, flags,
                                             base_index))

    def uniq_wait(self, slot: int, n: int, total: int, *, want_bytes=True, aligned=False):
        nbytes = self.out_arena_bytes(total, n) if aligned else total
        out = np.zeros(max(nbytes, 1), dtype=np.uint8) if want_bytes else None
        lens = np.zeros(max(n, 1), dtype=np.uint32)
        h = np.zeros(max(n, 1), dtype=np.uint64)
        first = np.zeros(max(n, 1), dtype=np.uint64)
        self._check(self._lib.ck_uniq_wait(self._h, slot, _ptr(out), _ptr(lens), _ptr(h), _ptr(first)))
        return dict(out=None if out is None else out[:nbytes], lens=lens[:n], hash=h[:n], first=first[:n])

    def uniq_wait_survivors(self, slot: int, n: int, total: int, *, want_bytes=True):
        """ck_uniq_wait_survivors (batch submitted with survivors=True): only what the first occurrences need crosses PCIe.
        -> dict(n_survivors, index[ns], offsets[ns + 1], bytes (compact arena), lens[n], hash[n], first[n])"""
        ns = C.c_uint32(0)
        index = np.zeros(max(n, 1), dtype=np.uint32)
        offs = np.zeros(max(n, 0) + 1, dtype=np.uint64)
        out = np.zeros(max(total + 16 * n, 1), dtype=np.uint8) if want_bytes else None
        lens = np.zeros(max(n, 1), dtype=np.uint32)
        h = np.zeros(max(n, 1), dtype=np.uint64)
        first = np.zeros(max(n, 1), dtype=np.uint64)
        self._check(self._lib.ck_uniq_wait_survivors(self._h, slot, C.byref(ns), _ptr(index), _ptr(offs), _ptr(out), _ptr(lens), _ptr(h),
                                                     _ptr(first)))
        k = int(ns.value)
        return dict(n_survivors=k, index=index[:k], offsets=offs[:k + 1], bytes=out, lens=lens[:n], hash=h[:n], first=first[:n])

    def mono_submit(self, slot: int, arena: np.ndarray, offsets: np.ndarray, opts: "N.CkMonoOptions", normalize: bool = True,
                    want_bytes: bool = True):
        """ck_mono_submit: `circkit monomerize`'s worker and consumer closures over a batch of raw record bytes"""
        flags = (N.CK_F_NORMALIZE if normalize else 0) | (0 if want_bytes else N.CK_F_NO_BYTES)
        self._check(self._lib.ck_mono_submit(self._h, slot, _ptr(arena), _ptr(offsets), len(offsets) - 1, flags, C.byref(opts)))

    def mono_wait(self, slot: int, n: int, total: int, want_bytes: bool = True):
        """ck_mono_wait -> dict(n_written, index[nw], offsets[nw + 1], bytes (compact arena), monomer_len[n], full_len[n],
        end[n] (CK_MONO_NONE = None))"""
        nw = C.c_uint32(0)
        index = np.zeros(max(n, 1), dtype=np.uint32)
        offs = np.zeros(max(n, 0) + 1, dtype=np.uint64)
        out = np.empty(max(total + 16 * n, 1), dtype=np.uint8) if want_bytes else None   # read only where written
        mono_len = np.zeros(max(n, 1), dtype=np.uint32)
        full_len = np.zeros(max(n, 1), dtype=np.uint32)
        end = np.zeros(max(n, 1), dtype=np.uint32)
        self._check(self._lib.ck_mono_wait(self._h, slot, C.byref(nw), _ptr(index), _ptr(offs), _ptr(out), _ptr(mono_len),
                                           _ptr(full_len), _ptr(end)))
        k = int(nw.value)
        return dict(n_written=k, index=index[:k], offsets=offs[:k + 1], bytes=out, monomer_len=mono_len[:n], full_len=full_len[:n],
                    end=end[:n])

    # -- FASTA text batches (ck_fasta_submit / ck_fasta_wait): record split, the command and the output framing on the device
    _COMMANDS = {"canonicalize": N.CK_CMD_CANONICALIZE, "uniq": N.CK_CMD_UNIQ, "monomerize": N.CK_CMD_MONOMERIZE}

    def fasta_out_bytes(self, text_bytes: int, n_records: int) -> int:
        return int(self._lib.ck_fasta_out_bytes(text_bytes, n_records))

    def fasta_submit(self, slot: int, text, command: str, *, base_index: int = 0, canonical_body: bool = False,
                     mono: "N.CkMonoOptions | None" = None) -> int:
        """ck_fasta_submit: `text` (bytes-like or a uint8 array, e.g. pinned) holds whole FASTA records and begins with '>';
        `command` is "canonicalize", "uniq" or "monomerize" (`mono`: mono_options).  -> number of records in the text"""
        a = text if isinstance(text, np.ndarray) else np.frombuffer(text, dtype=np.uint8)
        n = C.c_uint32(0)
        flags = N.CK_F_CANONICAL_BODY if canonical_body else 0
        rc = self._lib.ck_fasta_submit(self._h, slot, a.ctypes.data if len(a) else None, len(a), self._COMMANDS[command], flags,
                                       base_index, C.byref(mono) if mono is not None else None, C.byref(n))
        self._check(rc)
        self._text_batch[slot] = (int(n.value), len(a))
        return int(n.value)

    def fasta_wait(self, slot: int, out: "np.ndarray | None" = None) -> dict:
        """ck_fasta_wait -> dict(fasta = the bytes the CLI writes for the batch, n_written, index[nw] (positions of the written
        records in the batch), head[n, 2] (head ranges in the text), first[n] (uniq), full_len[n] / monomer_len[n]
        (monomerize)).  `out`: optional uint8 buffer (pinned, for speed) of at least fasta_out_bytes(text_bytes, n) bytes."""
        n, text_bytes = self._text_batch.pop(slot, (0, 0))
        need = self.fasta_out_bytes(text_bytes, n)
        if out is None or len(out) < need:
            out = np.empty(need, dtype=np.uint8)
        nbytes, nw = C.c_uint64(0), C.c_uint32(0)
        index = np.zeros(max(n, 1), dtype=np.uint32)
        head = np.zeros((max(n, 1), 2), dtype=np.uint64)
        first = np.zeros(max(n, 1), dtype=np.uint64)
        full_len = np.zeros(max(n, 1), dtype=np.uint32)
        mono_len = np.zeros(max(n, 1), dtype=np.uint32)
        self._check(self._lib.ck_fasta_wait(self._h, slot, out.ctypes.data, C.byref(nbytes), C.byref(nw), _ptr(index), _ptr(head),
                                            _ptr(first), _ptr(full_len), _ptr(mono_len)))
        k = int(nw.value)
        return dict(fasta=out[:int(nbytes.value)].tobytes(), n_written=k, index=index[:k], head=head[:n], first=first[:n],
                    full_len=full_len[:n], monomer_len=mono_len[:n])

    # -- DEFLATE on the device (ck_deflate_submit / ck_deflate_wait): raw, sync-flushed fragments of one deflate stream
    def deflate_bound(self, n: int) -> int:
        return int(self._lib.ck_deflate_bound(n))

    def deflate_submit(self, slot: int, data, dict=b"", crc: int = 0):
        """ck_deflate_submit: `data` (bytes-like or a uint8 array, e.g. pinned; 1 .. CK_DEFLATE_MAX_BYTES bytes) after `dict`
        (<= 32 KiB: the bytes that came before it in the stream); crc = the CRC-32 of everything before `data`"""
        a = data if isinstance(data, np.ndarray) else np.frombuffer(data, dtype=np.uint8)
        d = dict if isinstance(dict, np.ndarray) else np.frombuffer(dict, dtype=np.uint8)
        self._check(self._lib.ck_deflate_submit(self._h, slot, a.ctypes.data if len(a) else None, len(a),
                                                d.ctypes.data if len(d) else None, len(d), crc & 0xFFFFFFFF))
        self._deflate_batch[slot] = (len(a), a, d)      # pinned inputs must outlive the copy

    def deflate_wait(self, slot: int, out: "np.ndarray | None" = None) -> "tuple[bytes, int]":
        """ck_deflate_wait -> (raw deflate bytes ending in 00 00 ff ff, CRC-32 continued from the submit's crc).
        `out`: optional uint8 buffer (pinned, for speed) of at least deflate_bound(n) bytes."""
        n = self._deflate_batch.pop(slot, (0, None, None))[0]
        need = self.deflate_bound(n)
        if out is None or len(out) < need:
            out = np.empty(need, dtype=np.uint8)
        nbytes, crc = C.c_uint64(0), C.c_uint32(0)
        self._check(self._lib.ck_deflate_wait(self._h, slot, out.ctypes.data, C.byref(nbytes), C.byref(crc)))
        return out[:int(nbytes.value)].tobytes(), int(crc.value)

    def deflate(self, data, dict=b"", crc: int = 0) -> "tuple[bytes, int]":
        """deflate_submit + deflate_wait on slot 0"""
        self.deflate_submit(0, data, dict, crc)
        return self.deflate_wait(0)

    # -- bzip2 on the device (ck_bzip2_submit / ck_bzip2_wait): the blocks of one bzip2 stream, as libbzip2 writes at level 9
    def bzip2_bound(self, n: int) -> int:
        return int(self._lib.ck_bzip2_bound(n))

    def bzip2_submit(self, slot: int, data, final: bool, bits: int = 0, nbits: int = 0, crc: int = 0):
        """ck_bzip2_submit: `data` (bytes-like or a uint8 array; 1 .. CK_BZIP2_MAX_BYTES bytes) is the stream from its first
        byte not yet in a written block; (bits, nbits) the pending bits before it (nbits < 8, in the low bits of `bits`);
        crc the combined CRC of the blocks before it.  `final` writes every block, ending the stream's last run."""
        a = data if isinstance(data, np.ndarray) else np.frombuffer(data, dtype=np.uint8)
        self._check(self._lib.ck_bzip2_submit(self._h, slot, a.ctypes.data if len(a) else None, len(a), 1 if final else 0,
                                              bits & 0xFF, nbits, crc & 0xFFFFFFFF))
        self._bzip2_batch[slot] = len(a)

    def bzip2_wait(self, slot: int, out: "np.ndarray | None" = None) -> "tuple[bytes, int, int, int, int]":
        """ck_bzip2_wait -> (whole bytes of the blocks written, consumed input bytes, pending bits, their count, combined
        CRC).  `out`: optional uint8 buffer (pinned, for speed) of at least bzip2_bound(n) bytes."""
        n = self._bzip2_batch.pop(slot, 0)
        need = self.bzip2_bound(n)
        if out is None or len(out) < need:
            out = np.empty(need, dtype=np.uint8)
        nbytes, consumed = C.c_uint64(0), C.c_uint64(0)
        bits, nbits, crc = C.c_uint32(0), C.c_uint32(0), C.c_uint32(0)
        self._check(self._lib.ck_bzip2_wait(self._h, slot, out.ctypes.data, C.byref(nbytes), C.byref(consumed),
                                            C.byref(bits), C.byref(nbits), C.byref(crc)))
        return (out[:int(nbytes.value)].tobytes(), int(consumed.value), int(bits.value), int(nbits.value),
                int(crc.value))

    def bzip2(self, data, final: bool, bits: int = 0, nbits: int = 0, crc: int = 0):
        """bzip2_submit + bzip2_wait on slot 0"""
        self.bzip2_submit(0, data, final, bits, nbits, crc)
        return self.bzip2_wait(0)

    def bzip2_stats(self, slot: int = 0) -> "tuple[list[float], int]":
        """ck_bzip2_stats of the last call: device ms of (RLE1 and cuts, BWT, MTF, tables, pack), BWT sort rounds"""
        ms, rounds = (C.c_float * 5)(), C.c_uint32(0)
        self._check(self._lib.ck_bzip2_stats(self._h, slot, ms, C.byref(rounds)))
        return list(ms), int(rounds.value)

    def uniq_batch(self, arena: np.ndarray, offsets: np.ndarray, base_index: int = 0, *, normalize: bool = False,
                   want_bytes=True, aligned=False):
        """Worker + consumer closures over a batch (src/uniq.rs:33-78): dict(out, lens, hash, first)."""
        arena = np.ascontiguousarray(arena, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        self.uniq_submit(0, arena, offsets, base_index, normalize=normalize, no_bytes=not want_bytes, aligned=aligned)
        return self.uniq_wait(0, len(offsets) - 1, int(offsets[-1]) if len(offsets) else 0, want_bytes=want_bytes,
                              aligned=aligned)

    # -- multi-GPU uniq (one process and one context per GPU; include/circkit_b200.h, "multi-GPU uniq")
    def peer_export(self, world: int, rank: int, max_records: int) -> bytes:
        """allocate this rank's exchange block, return its CUDA IPC handle (give every rank the list of all of them)"""
        h = C.create_string_buffer(N.CK_PEER_HANDLE_BYTES)
        self._check(self._lib.ck_peer_export(self._h, world, rank, max_records, h))
        return h.raw

    def peer_attach(self, handles: "list[bytes]"):
        """map every rank's exchange block (handles in rank order); afterwards uniq submits are collective rounds"""
        blob = b"".join(handles)
        self._check(self._lib.ck_peer_attach(self._h, blob))

    def uniq_reset(self):
        self._check(self._lib.ck_uniq_reset(self._h))

    def uniq_grow(self, max_keys: Optional[int] = None):
        """ck_uniq_grow: the uniq table grows on the device as distinct keys arrive, up to max_keys keys (None: as many as
        device memory allows; 0: growth off)"""
        self._check(self._lib.ck_uniq_grow(self._h, 2**64 - 1 if max_keys is None else max_keys))

    def table_info(self) -> "tuple[int, int, int]":
        """ck_uniq_table_info -> (distinct keys in the table, keys it holds at 2/3 load, growths so far)"""
        keys, cap, grows = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        self._check(self._lib.ck_uniq_table_info(self._h, C.byref(keys), C.byref(cap), C.byref(grows)))
        return int(keys.value), int(cap.value), int(grows.value)


_default: Optional[Context] = None


def default_context() -> Context:
    global _default
    if _default is None:
        _default = Context(max_batch_bytes=1 << 20, max_batch_records=1 << 12)
    return _default


def lmsr_index(s: bytes) -> int:
    """lib/src/canonicalize.rs:5 -- index of the lexicographically minimal rotation (smallest on ties)."""
    return default_context().lmsr_index(bytes(s))


def lmsr(s: bytes) -> bytes:
    """lib/src/canonicalize.rs:41"""
    return default_context().lmsr(bytes(s))


def canonicalize(s: bytes) -> bytes:
    """lib/src/canonicalize.rs:54 -- min(lmsr(s), lmsr(revcomp(s))), ties keep the reverse complement."""
    return default_context().canonicalize(bytes(s))
