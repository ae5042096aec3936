"""`circkit canonicalize` / `circkit uniq` / `circkit monomerize` on the B200 path: the host side of the CLI drivers.

    python -m circkit_b200 canonicalize [INPUT] [-o OUTPUT] [-t THREADS]
    python -m circkit_b200 uniq [INPUT] [-o OUTPUT] [-c] [--table TABLE] [-t THREADS]
    python -m circkit_b200 monomerize [INPUT] [-o OUTPUT] [--seed-length N] [--max-mismatch N | --min-identity F] ... [--table TABLE]

Mirrors src/canonicalize.rs:7-51, src/uniq.rs:15-88 and src/monomerize.rs:16-160 with the flags of src/commands.rs:19-149.
The host reads (with the compression sniffing of src/utils.rs:9-27), cuts the decompressed text into pieces and batches of
whole records at '\n>' boundaries, writes (output compression by suffix, src/utils.rs:29-72) and builds the --table rows;
each batch of FASTA text goes to the C ABI's text entries (ck_fasta_submit / ck_fasta_wait, two slots in flight), where
seq_io 0.3.2's record split, normalisation, LMSR, the canonical form, XXH3-64, the first-occurrence table, the monomer
search and its filters, and the framing of the written records ('>' head '\n' body '\n', src/canonicalize.rs:33-37,
src/uniq.rs:50-61) run on the GPU.  What comes back is the bytes to write, plus the head ranges, first indices and
lengths the id checks and the tables need.  Input and output stream in pieces of 64 MB, so files larger than host memory
pass through.  Nothing is printed on success (tests/canon_uniq.rs:74-77); an I/O error exits non-zero with the OS message
on stderr.

`Records` and `_assemble` state the record split and the framing on the host (seq_io's rules, vectorised with numpy).
"""
from __future__ import annotations

import argparse
import bz2
import ctypes
import ctypes.util
import gzip
import lzma
import os
import struct
import sys

import numpy as np

from . import _native as N
from .core import Context


class FastaError(ValueError):
    pass


# ------------------------------------------------------------------------------------------------ (de)compression
def _zstd():
    name = ctypes.util.find_library("zstd") or "libzstd.so.1"
    lib = ctypes.CDLL(name)
    lib.ZSTD_getFrameContentSize.restype = ctypes.c_ulonglong
    lib.ZSTD_getFrameContentSize.argtypes = [ctypes.c_void_p, ctypes.c_size_t]
    lib.ZSTD_decompress.restype = ctypes.c_size_t
    lib.ZSTD_decompress.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t]
    lib.ZSTD_compressBound.restype = ctypes.c_size_t
    lib.ZSTD_compressBound.argtypes = [ctypes.c_size_t]
    lib.ZSTD_compress.restype = ctypes.c_size_t
    lib.ZSTD_compress.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]
    lib.ZSTD_isError.restype = ctypes.c_uint
    lib.ZSTD_isError.argtypes = [ctypes.c_size_t]
    return lib


def _zstd_decompress(raw: bytes) -> bytes:
    lib = _zstd()
    size = lib.ZSTD_getFrameContentSize(raw, len(raw))
    if size in (2**64 - 1, 2**64 - 2):                  # error / unknown size: grow until it fits
        size = max(4 * len(raw), 1 << 20)
    while True:
        buf = ctypes.create_string_buffer(int(size) or 1)
        got = lib.ZSTD_decompress(buf, len(buf), raw, len(raw))
        if not lib.ZSTD_isError(got):
            return buf.raw[:got]
        if size > (1 << 36):
            raise OSError("zstd: cannot decompress input")
        size *= 4


def _zstd_compress(data: bytes, level: int) -> bytes:
    lib = _zstd()
    buf = ctypes.create_string_buffer(lib.ZSTD_compressBound(len(data)) or 1)
    got = lib.ZSTD_compress(buf, len(buf), data, len(data), level)
    if lib.ZSTD_isError(got):
        raise OSError("zstd: cannot compress output")
    return buf.raw[:got]


def read_input(path: str | None) -> bytes:
    """src/utils.rs:9-27: file or stdin (refused when it is a terminal), format sniffed from the magic bytes (niffler)."""
    if path is None:
        if sys.stdin.isatty():
            raise OSError("No input file specified and stdin is a terminal")
        raw = sys.stdin.buffer.read()
    else:
        with open(path, "rb") as f:
            raw = f.read()
    if raw[:2] == b"\x1f\x8b":
        return gzip.decompress(raw)
    if raw[:3] == b"BZh":
        return bz2.decompress(raw)
    if raw[:6] == b"\xfd7zXZ\x00":
        return lzma.decompress(raw)
    if raw[:4] == b"\x28\xb5\x2f\xfd":
        return _zstd_decompress(raw)
    return raw


def write_output(path: str | None, data: bytes) -> None:
    """src/utils.rs:29-72: stdout, or a file compressed by its suffix (gz 6, bz2 9, xz 6, zst 1; anything else plain)."""
    if path is None:
        sys.stdout.buffer.write(data)
        sys.stdout.buffer.flush()
        return
    ext = path.rsplit(".", 1)[-1] if "." in os.path.basename(path) else ""
    if ext == "gz":
        data = gzip.compress(data, compresslevel=6)
    elif ext == "bz2":
        data = bz2.compress(data, compresslevel=9)
    elif ext == "xz":
        data = lzma.compress(data, preset=6)
    elif ext == "zst":
        data = _zstd_compress(data, 1)
    with open(path, "wb") as f:
        f.write(data)


# ------------------------------------------------------------------------------------------------ FASTA records
class Records:
    """Record boundaries of a FASTA buffer as index arrays (seq_io 0.3.2 `fasta::Reader` rules): a record starts at a
    '>' that follows a '\\n'; head = header line without '>' and one trailing '\\r'; seq = everything between the
    header's '\\n' and the record's last '\\n' (or EOF), internal line breaks included, one trailing '\\r' trimmed."""

    def __init__(self, data: bytes):
        d = np.frombuffer(data, dtype=np.uint8)
        n = len(d)
        self.data = d
        nl = np.flatnonzero(d == 10)
        # leading empty lines ("" or "\r") are skipped; the first other line must start with '>'
        pos = 0
        while pos < n:
            k = int(np.searchsorted(nl, pos))
            end = int(nl[k]) if k < len(nl) else n
            line_len = end - pos
            if not (line_len == 0 or (line_len == 1 and d[pos] == 13)):
                break
            if k >= len(nl):
                pos = n
                break
            pos = end + 1
        empty = np.zeros(0, dtype=np.int64)
        if pos >= n:
            self.head_lo = self.head_hi = self.seq_lo = self.seq_hi = empty
            return
        if d[pos] != ord(">"):
            raise FastaError("expected '>' at record start")
        gt = np.flatnonzero(d == ord(">"))
        gt = gt[gt > pos]
        starts = np.concatenate([[pos], gt[d[gt - 1] == 10]]).astype(np.int64)
        # region end: the '\n' before the next record's '>' (excluded), else EOF without one final '\n'
        last_end = n - 1 if d[n - 1] == 10 else n
        region_end = np.concatenate([starts[1:] - 1, [last_end]]).astype(np.int64)
        if len(nl):
            k = np.searchsorted(nl, starts)
            first_nl = np.where(k < len(nl), nl[np.minimum(k, len(nl) - 1)], n).astype(np.int64)
        else:
            first_nl = np.full(len(starts), n, dtype=np.int64)
        has_seq = first_nl < region_end
        head_hi = np.where(has_seq, first_nl, region_end)
        head_lo = starts + 1
        head_hi = np.maximum(head_hi, head_lo)
        cr = (head_hi > head_lo) & (d[np.maximum(head_hi - 1, 0)] == 13)
        self.head_lo, self.head_hi = head_lo, head_hi - cr
        seq_lo = np.where(has_seq, first_nl + 1, region_end)
        seq_hi = np.maximum(region_end, seq_lo)
        cr = (seq_hi > seq_lo) & (d[np.maximum(seq_hi - 1, 0)] == 13)
        self.seq_lo, self.seq_hi = seq_lo, seq_hi - cr

    def __len__(self):
        return len(self.head_lo)

    def gather(self, lo: np.ndarray, hi: np.ndarray) -> np.ndarray:
        """concatenation of data[lo[i]:hi[i]] over i (regions are disjoint and increasing)"""
        return self.data[_region_mask(len(self.data), lo, hi)]

    def ids(self) -> list[bytes]:
        """record.id(): head up to the first ' ' (src/uniq.rs:48,67 unwrap it as UTF-8)"""
        out = []
        for a, b in zip(self.head_lo.tolist(), self.head_hi.tolist()):
            h = self.data[a:b].tobytes().split(b" ", 1)[0]
            h.decode("utf-8")
            out.append(h)
        return out


def _region_mask(n: int, lo: np.ndarray, hi: np.ndarray) -> np.ndarray:
    delta = np.zeros(n + 1, dtype=np.int32)
    np.add.at(delta, lo, 1)
    np.add.at(delta, hi, -1)
    return np.cumsum(delta[:-1]) > 0


def _assemble(heads: np.ndarray, head_len: np.ndarray, bodies: np.ndarray, body_len: np.ndarray) -> bytes:
    """'>' head '\\n' body '\\n' for every record (src/canonicalize.rs:33-37), from the concatenated heads / bodies."""
    m = len(head_len)
    if m == 0:
        return b""
    rec_len = head_len + body_len + 3
    start = np.zeros(m + 1, dtype=np.int64)
    np.cumsum(rec_len, out=start[1:])
    out = np.empty(int(start[-1]), dtype=np.uint8)
    out[start[:-1]] = ord(">")
    out[start[:-1] + 1 + head_len] = 10
    out[start[1:] - 1] = 10
    out[_region_mask(len(out), start[:-1] + 1, start[:-1] + 1 + head_len)] = heads
    out[_region_mask(len(out), start[:-1] + 2 + head_len, start[1:] - 1)] = bodies
    return out.tobytes()


# ------------------------------------------------------------------------------------------------ streaming I/O
CHUNK_BYTES = 64 << 20


class _ZstdReader:
    """streaming zstd decompression through libzstd (no Python module in the image): file-like .read(n)"""

    def __init__(self, f):
        name = ctypes.util.find_library("zstd") or "libzstd.so.1"
        self.lib = lib = ctypes.CDLL(name)
        lib.ZSTD_createDStream.restype = ctypes.c_void_p
        lib.ZSTD_freeDStream.argtypes = [ctypes.c_void_p]
        lib.ZSTD_decompressStream.restype = ctypes.c_size_t
        lib.ZSTD_decompressStream.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        lib.ZSTD_isError.restype = ctypes.c_uint
        lib.ZSTD_isError.argtypes = [ctypes.c_size_t]
        self.f, self.ds, self.src, self.pos, self.eof = f, lib.ZSTD_createDStream(), b"", 0, False

    def read(self, n: int) -> bytes:
        class Buf(ctypes.Structure):
            _fields_ = [("p", ctypes.c_void_p), ("size", ctypes.c_size_t), ("pos", ctypes.c_size_t)]
        out = ctypes.create_string_buffer(n)
        ob = Buf(ctypes.cast(out, ctypes.c_void_p), n, 0)
        while ob.pos < n:
            if self.pos >= len(self.src):
                if self.eof:
                    break
                self.src, self.pos = self.f.read(1 << 20), 0
                if not self.src:
                    self.eof = True
                    break
            keep = ctypes.create_string_buffer(self.src, len(self.src))
            ib = Buf(ctypes.cast(keep, ctypes.c_void_p), len(self.src), self.pos)
            rc = self.lib.ZSTD_decompressStream(self.ds, ctypes.byref(ob), ctypes.byref(ib))
            if self.lib.ZSTD_isError(rc):
                raise OSError("zstd: cannot decompress input")
            self.pos = ib.pos
        return out.raw[:ob.pos]

    def close(self):
        if self.ds:
            self.lib.ZSTD_freeDStream(self.ds)
            self.ds = None


def iter_input(path: str | None, chunk_bytes: int = CHUNK_BYTES):
    """src/utils.rs:9-27 as a stream: decompressed chunks of the input (format sniffed from the magic bytes), so that a file
    far larger than host memory passes through"""
    if path is None:
        if sys.stdin.isatty():
            raise OSError("No input file specified and stdin is a terminal")
        f = sys.stdin.buffer
    else:
        f = open(path, "rb")
    try:
        import io
        head = f.peek(8)[:8] if hasattr(f, "peek") else b""
        if not head and not hasattr(f, "peek"):
            f = io.BufferedReader(f)
            head = f.peek(8)[:8]
        if head[:2] == b"\x1f\x8b":
            r = gzip.GzipFile(fileobj=f)
        elif head[:3] == b"BZh":
            r = bz2.BZ2File(f)
        elif head[:6] == b"\xfd7zXZ\x00":
            r = lzma.LZMAFile(f)
        elif head[:4] == b"\x28\xb5\x2f\xfd":
            r = _ZstdReader(f)
        else:
            r = f
        while True:
            c = r.read(chunk_bytes)
            if not c:
                break
            yield c
    finally:
        if path is not None:
            f.close()


def _suffix(path: str | None) -> str:
    return path.rsplit(".", 1)[-1] if path is not None and "." in os.path.basename(path) else ""


# one gzip member (RFC 1952) with no name, mtime 0 and OS unknown, so that the same output gives the same file
GZIP_HEADER = b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\xff"


class DeviceDeflate:
    """Raw DEFLATE on the GPU for Writer's gzip output (ck_deflate_submit / ck_deflate_wait): deflate(data, dict, crc) ->
    (fragment, crc) compresses up to max_bytes bytes after `dict` (the <= 32 KiB before them) into blocks that end with a
    sync flush (00 00 ff ff), and continues the CRC-32.  The context (no batch staging, so the pump's slots are untouched)
    and the pinned buffers are created by the first call."""

    max_bytes = N.CK_DEFLATE_MAX_BYTES

    def __init__(self, device: int = 0):
        self.device, self.ctx, self.pinned = device, None, {}

    def _buf(self, which: int, size: int) -> np.ndarray:
        p = self.pinned.get(which)
        if p is None or len(p[1]) < size:
            if p is not None:
                self.ctx._lib.ck_free_pinned(self.ctx.handle, p[0])
            size = (size + (16 << 20) - 1) & ~((16 << 20) - 1)
            ptr = self.ctx._lib.ck_alloc_pinned(self.ctx.handle, size)
            if not ptr:
                raise MemoryError("cannot allocate %d bytes of pinned host memory" % size)
            p = (ptr, np.ctypeslib.as_array((ctypes.c_uint8 * size).from_address(ptr)))
            self.pinned[which] = p
        return p[1]

    def deflate(self, data, dict: bytes, crc: int) -> "tuple[bytes, int]":
        if self.ctx is None:
            self.ctx = Context(self.device, max_batch_bytes=0, max_batch_records=0)
        n = len(data)
        src = self._buf(0, n)[:n]
        src[:] = np.frombuffer(data, dtype=np.uint8)
        out = self._buf(1, self.ctx.deflate_bound(n))
        self.ctx.deflate_submit(0, src, dict, crc)
        return self.ctx.deflate_wait(0, out)

    def close(self):
        if self.ctx is not None:
            for p, _ in self.pinned.values():
                self.ctx._lib.ck_free_pinned(self.ctx.handle, p)
            self.pinned = {}
            self.ctx.close()
            self.ctx = None


class Writer:
    """src/utils.rs:29-72 as a stream: stdout, or a file compressed by its suffix (gz 6, bz2 9, xz 6, zst 1; else plain).
    gzip_encoder (gz only; e.g. DeviceDeflate()): an object with max_bytes, deflate(data, dict, crc) -> (raw deflate
    fragment ending in a sync flush, crc) and close().  Writer then frames the gzip member itself: GZIP_HEADER, one
    fragment per call of at most max_bytes bytes, each given the last 32 KiB written before it as its dictionary, and at
    close the final empty block (03 00), the CRC-32 and ISIZE.  Without it, gz goes through gzip.GzipFile at level 6."""

    def __init__(self, path: str | None, gzip_encoder=None):
        self.path, self.zst, self.gz = path, None, None
        if path is None:
            self.f = sys.stdout.buffer
            return
        ext = _suffix(path)
        if ext == "gz" and gzip_encoder is not None:
            self.f, self.gz = open(path, "wb"), gzip_encoder
            self.crc, self.size, self.tail = 0, 0, b""
            self.f.write(GZIP_HEADER)
        elif ext == "gz":
            self.f = gzip.GzipFile(path, "wb", compresslevel=6)
        elif ext == "bz2":
            self.f = bz2.BZ2File(path, "wb", compresslevel=9)
        elif ext == "xz":
            self.f = lzma.LZMAFile(path, "wb", preset=6)
        elif ext == "zst":
            self.f, self.zst = open(path, "wb"), []          # libzstd one-shot frames: one frame per written piece
        else:
            self.f = open(path, "wb")

    def write(self, data: bytes):
        if not data:
            return
        if self.gz is not None:
            mv = memoryview(data).cast("B")
            for lo in range(0, len(mv), self.gz.max_bytes):
                piece = mv[lo:lo + self.gz.max_bytes]
                frag, self.crc = self.gz.deflate(piece, self.tail, self.crc)
                self.f.write(frag)
                self.size += len(piece)
                self.tail = (self.tail + piece[-32768:].tobytes())[-32768:]
        elif self.zst is not None:
            self.f.write(_zstd_compress(data, 1))             # concatenated frames are one valid zstd stream
        else:
            self.f.write(data)

    def close(self):
        if self.path is None:
            self.f.flush()
            return
        try:
            if self.gz is not None:                          # final empty fixed block, CRC-32, ISIZE (RFC 1952)
                self.f.write(b"\x03\x00" + struct.pack("<II", self.crc, self.size & 0xFFFFFFFF))
        finally:
            try:
                if self.gz is not None:
                    self.gz.close()
            finally:
                self.f.close()


def iter_text(chunks):
    """Pieces of whole records over a stream of chunks: each piece is cut before the last '\\n>' of what has been read (the
    record that follows may be unfinished and is carried into the next piece).  Every piece but the first begins with '>';
    the first keeps seq_io's leading blank lines (see _piece_text)."""
    carry = b""
    first = True
    for c in chunks:
        data = carry + c if carry else c
        cut = data.rfind(b"\n>") + 1
        if cut == 0:                                         # no record start after the first byte: keep accumulating
            carry = data
            continue
        piece, carry = data[:cut], data[cut:]
        if not first and piece[:1] != b">":
            raise FastaError("expected '>' at record start")
        first = False
        yield piece
    if carry or first:
        yield carry


def iter_records(chunks):
    """Records objects over a stream of chunks, cut as iter_text cuts them: every yield holds whole records only.  seq_io's
    leading-blank-line rule applies to the first piece only."""
    for piece in iter_text(chunks):
        yield Records(piece)


def _piece_text(piece) -> bytes:
    """the text of a piece from its first record's '>' on: a Records piece's data, or a text piece of iter_text with seq_io's
    leading empty lines ("" or "\\r") skipped; any other first line -> FastaError"""
    if isinstance(piece, Records):
        return piece.data[int(piece.head_lo[0]) - 1:].tobytes() if len(piece) else b""
    pos, n = 0, len(piece)
    while pos < n and piece[pos] != 62:
        end = piece.find(b"\n", pos)
        if piece[pos:end if end >= 0 else n] not in (b"", b"\r"):
            raise FastaError("expected '>' at record start")
        pos = n if end < 0 else end + 1
    return piece[pos:] if pos else piece


# ------------------------------------------------------------------------------------------------ GPU pump
MAX_BATCH_BYTES = 256 << 20
MAX_BATCH_RECORDS = 1 << 20
# distinct records uniq's table holds when it is created (about 25 MB of device memory); it grows on the device as they arrive
UNIQ_TABLE_KEYS = 1 << 20


def _text_batches(text: bytes, max_bytes: int, max_records: int, oversize: bool = False):
    """(lo, hi) cuts of a piece of whole records (text[0] == '>') at '\\n>' boundaries, each of at most max_bytes bytes and
    max_records records; a record longer than max_bytes is a cut of its own with oversize=True, else a FastaError"""
    n, lo = len(text), 0
    while lo < n:
        hi = n if n - lo <= max_bytes else text.rfind(b"\n>", lo, lo + max_bytes + 1) + 1
        if hi <= lo:
            if not oversize:
                raise FastaError("record longer than the batch size")
            hi = text.find(b"\n>", lo) + 1 or n
        if text.count(b"\n>", lo, hi) >= max_records:       # more records than a batch takes: cut after max_records of them
            d = np.frombuffer(text, dtype=np.uint8, count=hi - lo, offset=lo)
            hi = lo + int(np.flatnonzero((d[:-1] == 10) & (d[1:] == 62))[max_records - 1]) + 1
        yield lo, hi
        lo = hi


def _context(table_capacity: int) -> Context:
    return Context(max_batch_bytes=MAX_BATCH_BYTES, max_batch_records=MAX_BATCH_RECORDS, table_capacity=table_capacity)


class _Pump:
    """Text batches through the two slots of a context (ck_fasta_submit / ck_fasta_wait): batch b is copied into slot
    b & 1's pinned buffer and submitted (the submit returns once the device has split it), then batch b - 1 is collected
    and handed to done(text, lo, result, base_index, tag); the record split, the command and the output framing run on the
    device.  Batches come from pieces fed in input order.  A record longer than MAX_BATCH_BYTES (monomerize: oversize=True)
    is a batch of its own on a second context sized for it."""

    def __init__(self, command: str, done, table_capacity: int = 0, oversize: bool = False, **submit_kw):
        self.command, self.done, self.oversize, self.kw = command, done, oversize, submit_kw
        self.ctx, self.big = _context(table_capacity), None
        if command == "uniq":
            self.ctx.uniq_grow()
        self.pinned = {}                                     # (slot, 0 in / 1 out) -> (pointer, uint8 array)
        self.pend, self.b, self.base = None, 0, 0

    def _buf(self, slot: int, which: int, size: int) -> np.ndarray:
        p = self.pinned.get((slot, which))
        if p is None or len(p[1]) < size:
            if p is not None:
                self.ctx._lib.ck_free_pinned(self.ctx.handle, p[0])
            size = (size + (16 << 20) - 1) & ~((16 << 20) - 1)
            ptr = self.ctx._lib.ck_alloc_pinned(self.ctx.handle, size)
            if not ptr:
                raise MemoryError("cannot allocate %d bytes of pinned host memory" % size)
            p = (ptr, np.ctypeslib.as_array((ctypes.c_uint8 * size).from_address(ptr)))
            self.pinned[(slot, which)] = p
        return p[1]

    def feed(self, text: bytes, tag=None):
        for lo, hi in _text_batches(text, MAX_BATCH_BYTES, MAX_BATCH_RECORDS, self.oversize):
            slot, size, ctx = self.b & 1, hi - lo, self.ctx
            if size > MAX_BATCH_BYTES:
                if self.big is None or self.big.max_batch_bytes < size:
                    if self.pend is not None and self.pend[0] is self.big:
                        self._finish()
                    if self.big is not None:
                        self.big.close()
                    self.big = Context(max_batch_bytes=size, max_batch_records=1)
                ctx = self.big
            buf = self._buf(slot, 0, size)[:size]
            buf[:] = np.frombuffer(text, dtype=np.uint8, count=size, offset=lo)
            n = ctx.fasta_submit(slot, buf, self.command, base_index=self.base, **self.kw)
            if self.pend is not None:
                self._finish()
            self.pend = (ctx, slot, text, lo, self.base, tag, ctx.fasta_out_bytes(size, n))
            self.base += n
            self.b += 1

    def _finish(self):
        ctx, slot, text, lo, base, tag, out_bytes = self.pend
        self.pend = None
        self.done(text, lo, ctx.fasta_wait(slot, self._buf(slot, 1, out_bytes)), base, tag)

    def close(self, ok: bool = True):
        try:
            if ok and self.pend is not None:
                self._finish()
        finally:
            for p, _ in self.pinned.values():
                self.ctx._lib.ck_free_pinned(self.ctx.handle, p)
            self.pinned = {}
            for c in (self.ctx, self.big):
                if c is not None:
                    c.close()


def _drive(pieces, command: str, done, piece_tag=None, **kw):
    """every piece's text through a _Pump (created at the first non-empty piece); piece_tag(text) goes to `done` with each
    of the piece's batches"""
    pump = None
    ok = False
    try:
        for piece in pieces:
            text = _piece_text(piece)
            if not text:
                continue
            if pump is None:
                pump = _Pump(command, done, **kw)
            pump.feed(text, piece_tag(text) if piece_tag else None)
        ok = True
    finally:
        if pump is not None:
            pump.close(ok)


def run_canonicalize(pieces, write, threads: int = 0) -> None:
    """`circkit canonicalize` over a stream of pieces (text pieces of iter_text or Records; src/canonicalize.rs:7-51):
    `write(bytes)` gets the output.  `threads` is accepted for the command line's sake: the host does no per-record work."""
    _drive(pieces, "canonicalize", lambda text, lo, r, base, tag: write(r["fasta"]))


def _csv_field(f: bytes, delim: bytes) -> bytes:
    """csv 1.2.2 defaults (QuoteStyle::Necessary, double_quote, terminator '\\n')"""
    if any(c in f for c in (delim, b'"', b"\n", b"\r")):
        return b'"' + f.replace(b'"', b'""') + b'"'
    return f


def _rec_id(text: bytes, lo: int, head: np.ndarray, i: int) -> bytes:
    """record.id(): head up to the first ' ' (src/uniq.rs:48,67 unwrap it as UTF-8)"""
    return text[lo + int(head[i, 0]): lo + int(head[i, 1])].split(b" ", 1)[0]


def run_uniq(pieces, write, canonical: bool = False, table_write=None, table_ext: str | None = None,
             table_capacity: int | None = None, threads: int = 0) -> None:
    """`circkit uniq` over a stream of pieces (src/uniq.rs:15-88): one first-occurrence table on the device for the whole
    input, survivors written batch by batch in input order, duplicate rows to `table_write` as they are met.
    `table_capacity`: the table's initial size in keys (default UNIQ_TABLE_KEYS); it grows as distinct records arrive."""
    if table_capacity is None:
        table_capacity = UNIQ_TABLE_KEYS
    first_ids = {}                                             # global index of a first occurrence -> its id (for --table only)
    delim = b"\t" if table_ext == "tsv" else b","
    state = {"header": False}

    def done(text, lo, r, base, ascii_text):
        head, keep_idx = r["head"], r["index"]
        if not ascii_text:                                     # record.id().unwrap(): survivors, or every record with --table
            for i in (range(len(head)) if table_write is not None else keep_idx.tolist()):
                _rec_id(text, lo, head, i).decode("utf-8")
        write(r["fasta"])
        if table_write is not None:                            # src/uniq.rs:62-71, csv 1.2.2 defaults
            for i in keep_idx.tolist():
                first_ids[base + i] = _rec_id(text, lo, head, i)
            keep = np.zeros(len(head), dtype=bool)
            keep[keep_idx] = True
            rows = bytearray()
            for i in np.flatnonzero(~keep).tolist():
                if not state["header"]:
                    rows += b"id" + delim + b"duplicate_id\n"
                    state["header"] = True
                rows += _csv_field(first_ids[int(r["first"][i])], delim) + delim + _csv_field(_rec_id(text, lo, head, i), delim) + b"\n"
            table_write(bytes(rows))

    _drive(pieces, "uniq", done, bytes.isascii, table_capacity=table_capacity, canonical_body=canonical)


def canonicalize(fasta: bytes) -> bytes:
    """bytes of a FASTA file -> bytes `circkit canonicalize` writes (src/canonicalize.rs:7-51)"""
    out = []
    run_canonicalize(iter_text([fasta] if fasta else []), out.append)
    return b"".join(out)


def uniq(fasta: bytes, canonical: bool = False, table_ext: str | None = None):
    """bytes of a FASTA file -> (bytes `circkit uniq` writes, bytes of the --table file or None) (src/uniq.rs:15-88)"""
    out, table = [], ([] if table_ext is not None else None)
    n_upper = fasta.count(b">") + 1
    run_uniq(iter_text([fasta] if fasta else []), out.append, canonical, table.append if table is not None else None, table_ext,
             table_capacity=n_upper)
    return b"".join(out), (b"".join(table) if table is not None else None)


class CliError(ValueError):
    """argument combinations the reference rejects with `bail!` (src/monomerize.rs:35-45)"""


def mono_options(sensitive: bool = False, seed_length: int = 10, max_mismatch=None, min_identity=None, min_overlap=None,
                 min_overlap_percent=None, min_length: int = 0, max_length=None, keep_all: bool = False):
    """the options of `circkit monomerize` (src/commands.rs:19-90) as ck_mono_options, checked like the CLI's bail!s
    (src/monomerize.rs:35-45) and the builder (lib/src/monomerize.rs:20-40) before anything touches the device"""
    from ._native import CK_MONO_KEEP_ALL, CK_MONO_SENSITIVE, CkMonoOptions
    if max_mismatch is not None and min_identity is not None:
        raise CliError("cannot specify both max_mismatch and min_identity")
    if min_identity is not None and not 0.0 <= min_identity <= 1.0:
        raise CliError("min_identity must be between 0.0 and 1.0")
    if not 1 <= seed_length <= 63:
        raise CliError("Seed length must be at least 1 and at most 63 but was set to %d." % seed_length)
    for name, v in (("max_mismatch", max_mismatch), ("min_overlap", min_overlap), ("min_length", min_length),
                    ("max_length", max_length)):
        if v is not None and v < 0:                          # usize in the reference
            raise CliError("%s must not be negative" % name)
    return CkMonoOptions(seed_length, (CK_MONO_SENSITIVE if sensitive else 0) | (CK_MONO_KEEP_ALL if keep_all else 0),
                         max_mismatch or 0, -1.0 if min_identity is None else float(min_identity), min_length,
                         2**64 - 1 if max_length is None else max_length, min_overlap or 0,
                         float("nan") if min_overlap_percent is None else float(min_overlap_percent))


def run_monomerize(pieces, write, opts, table_write=None, table_ext: str | None = None) -> None:
    """`circkit monomerize` over a stream of pieces (src/monomerize.rs:16-160): `opts` from mono_options; normalisation,
    the monomer search, the length / overlap filters of the consumer closure, the extraction of full_seq[..end] and the
    framing run on the device; `write(bytes)` gets the output ('>' head '\\n' monomer '\\n'), `table_write` the --table rows
    as batches complete."""
    delim = b"\t" if table_ext == "tsv" else b","
    state = {"header": False}

    def done(text, lo, r, base, tag):
        write(r["fasta"])
        if table_write is not None and r["n_written"]:       # :145-154, csv 1.2.2 defaults: header with the first row
            rows = bytearray()
            if not state["header"]:
                rows += delim.join([b"id", b"original_length", b"monomer_length"]) + b"\n"
                state["header"] = True
            head, full_len, mono_len = r["head"], r["full_len"], r["monomer_len"]
            for i in r["index"].tolist():
                h = text[lo + int(head[i, 0]): lo + int(head[i, 1])]
                h.decode("utf-8")                             # std::str::from_utf8(record.head()).unwrap()
                rows += delim.join([_csv_field(h, delim), b"%d" % full_len[i], b"%d" % mono_len[i]]) + b"\n"
            table_write(bytes(rows))

    _drive(pieces, "monomerize", done, oversize=True, mono=opts)


def monomerize(fasta: bytes, sensitive: bool = False, seed_length: int = 10, max_mismatch=None, min_identity=None,
               min_overlap=None, min_overlap_percent=None, min_length: int = 0, max_length=None, keep_all: bool = False,
               table_ext: str | None = None):
    """bytes of a FASTA file -> (bytes `circkit monomerize` writes, bytes of the --table file or None)
    (src/monomerize.rs:16-160), through run_monomerize"""
    opts = mono_options(sensitive, seed_length, max_mismatch, min_identity, min_overlap, min_overlap_percent, min_length,
                        max_length, keep_all)
    out, table = [], ([] if table_ext is not None else None)
    run_monomerize(iter_text([fasta] if fasta else []), out.append, opts, table.append if table is not None else None, table_ext)
    return b"".join(out), (b"".join(table) if table is not None else None)


# ------------------------------------------------------------------------------------------------ entry point
def main(argv=None) -> int:
    ap = argparse.ArgumentParser(prog="circkit", description="canonicalize / uniq on the B200 path")
    ap.add_argument("-v", "--verbose", action="count", default=0)
    ap.add_argument("-q", "--quiet", action="count", default=0)
    sub = ap.add_subparsers(dest="command", required=True)
    c = sub.add_parser("canonicalize", aliases=["canon"])
    c.add_argument("input", nargs="?")
    c.add_argument("-o", "--output")
    c.add_argument("-t", "--threads", type=int, default=os.cpu_count())
    u = sub.add_parser("uniq")
    u.add_argument("input", nargs="?")
    u.add_argument("-o", "--output")
    u.add_argument("-c", "--canonicalize", "--norm", "--canon", dest="canonicalize", action="store_true")
    u.add_argument("--table")
    u.add_argument("-t", "--threads", type=int, default=os.cpu_count())
    mo = sub.add_parser("monomerize")                          # src/commands.rs:19-90
    mo.add_argument("input", nargs="?")
    mo.add_argument("-o", "--output")
    mo.add_argument("--sensitive", action="store_true")
    mo.add_argument("--seed-length", type=int, default=10, choices=range(5, 65), metavar="[5..64]")
    mo.add_argument("--max-mismatch", type=int)
    mo.add_argument("--min-identity", type=float)
    mo.add_argument("--min-overlap", type=int)
    mo.add_argument("--min-overlap-percent", type=float)
    mo.add_argument("--min-length", type=int, default=0)
    mo.add_argument("--max-length", type=int)
    mo.add_argument("-k", "--keep-all", action="store_true")
    mo.add_argument("--table")
    mo.add_argument("-t", "--threads", type=int, default=os.cpu_count())
    mo.add_argument("--batch-size", type=int, default=64, help=argparse.SUPPRESS)
    args = ap.parse_args(argv)
    try:
        threads = max(1, args.threads or 1)
        opts = None
        if args.command == "monomerize":                      # argument errors before any file is opened
            opts = mono_options(args.sensitive, args.seed_length, args.max_mismatch, args.min_identity, args.min_overlap,
                                args.min_overlap_percent, args.min_length, args.max_length, args.keep_all)
        # every subcommand streams: decompress, cut into pieces of whole records, process and write batch by batch
        # (src/utils.rs:9-72); the record split is the device's
        pieces = iter_text(iter_input(args.input))
        first = next(pieces, None)                              # open the input (and fail on it) before the output is created
        if first is not None:
            first = _piece_text(first)

        def chain():
            if first is not None:
                yield first
            yield from pieces
        w = Writer(args.output, gzip_encoder=DeviceDeflate() if _suffix(args.output) == "gz" else None)
        tf = None
        try:
            ext = None
            if getattr(args, "table", None) is not None:           # uniq / monomerize --table
                ext = "tsv" if args.table.endswith(".tsv") else "csv"
                tf = open(args.table, "wb")
            if args.command in ("canonicalize", "canon"):
                run_canonicalize(chain(), w.write, threads=threads)
            elif args.command == "monomerize":
                run_monomerize(chain(), w.write, opts, tf.write if tf else None, ext)
            else:
                run_uniq(chain(), w.write, args.canonicalize, tf.write if tf else None, ext, threads=threads)
        finally:
            w.close()
            if tf is not None:
                tf.close()
    except OSError as e:
        msg = e.strerror or str(e)
        print("Error: %s%s" % (msg, " (os error %d)" % e.errno if e.errno else ""), file=sys.stderr)
        return 1
    except (FastaError, UnicodeDecodeError, CliError, ValueError) as e:
        print("Error: %s" % e, file=sys.stderr)
        return 1
    return 0
