"""`circkit canonicalize` / `circkit uniq` / `circkit monomerize` on the B200 path: the host side of the CLI drivers.

    python -m circkit_b200 canonicalize [INPUT] [-o OUTPUT] [-t THREADS]
    python -m circkit_b200 uniq [INPUT] [-o OUTPUT] [-c] [--table TABLE] [-t THREADS]
    python -m circkit_b200 monomerize [INPUT] [-o OUTPUT] [--seed-length N] [--max-mismatch N | --min-identity F] ... [--table TABLE]

Mirrors src/canonicalize.rs:7-51 and src/uniq.rs:15-88 with the flags of src/commands.rs:112-149: the host keeps what
the reference keeps on the host -- reading (with the compression sniffing of src/utils.rs:9-27), FASTA record splitting
(seq_io 0.3.2 rules), writing in the reference's framing (src/canonicalize.rs:33-37, src/uniq.rs:50-61), the duplicate
table (src/uniq.rs:62-71, src/utils.rs:74-84) and output compression by suffix (src/utils.rs:29-72) -- and hands batches
of record bytes, packed to 2 bits per base by `--threads` host threads (ck_pack2_host), to the C ABI (ck_*_submit_packed,
two slots in flight), where LMSR, the canonical form, XXH3-64, the first-occurrence table and the compaction of the
survivors run on the GPU.  `monomerize` (src/monomerize.rs:16-160) hands the raw record bytes to ck_mono_submit /
ck_mono_wait the same way; normalisation, the monomer search, the length / overlap filters and the extraction of the written
monomers run on the GPU.  Input and output stream in pieces of 64 MB, so files larger than host memory pass through.
Nothing is printed on success (tests/canon_uniq.rs:74-77); an I/O error exits non-zero with the OS message on stderr.

Record splitting and output assembly are numpy-vectorised (no per-record Python on the canonicalize path).
"""
from __future__ import annotations

import argparse
import bz2
import ctypes
import ctypes.util
import gzip
import lzma
import os
import sys

import numpy as np

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


class Writer:
    """src/utils.rs:29-72 as a stream: stdout, or a file compressed by its suffix (gz 6, bz2 9, xz 6, zst 1; else plain)"""

    def __init__(self, path: str | None):
        self.path, self.zst = path, None
        if path is None:
            self.f = sys.stdout.buffer
            return
        ext = path.rsplit(".", 1)[-1] if "." in os.path.basename(path) else ""
        if ext == "gz":
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
        if self.zst is not None:
            self.f.write(_zstd_compress(data, 1))             # concatenated frames are one valid zstd stream
        else:
            self.f.write(data)

    def close(self):
        if self.path is None:
            self.f.flush()
        else:
            self.f.close()


def iter_records(chunks):
    """Records objects over a stream of chunks: every yield holds whole records only (the tail of a chunk that may belong to
    an unfinished record is carried into the next one).  seq_io's leading-blank-line rule applies to the first piece only."""
    carry = b""
    first = True
    for c in chunks:
        data = carry + c if carry else c
        d = np.frombuffer(data, dtype=np.uint8)
        gt = np.flatnonzero(d == ord(">"))
        gt = gt[(gt > 0)]
        gt = gt[d[gt - 1] == 10]
        if len(gt) == 0:                                     # no record start after the first byte: keep accumulating
            carry = data
            continue
        cut = int(gt[-1])                                    # the last record of the piece may be unfinished: hold it back
        piece, carry = data[:cut], data[cut:]
        if not first and piece[:1] != b">":
            raise FastaError("expected '>' at record start")
        first = False
        yield Records(piece)
    if carry or first:
        yield Records(carry)


# ------------------------------------------------------------------------------------------------ GPU pump
MAX_BATCH_BYTES = 256 << 20
MAX_BATCH_RECORDS = 1 << 20


def _batches(offsets: np.ndarray, oversize: bool = False):
    """cuts of the record range into batches of <= MAX_BATCH_BYTES / MAX_BATCH_RECORDS; oversize=True: a record longer than
    MAX_BATCH_BYTES is a batch of its own (else FastaError)"""
    n = len(offsets) - 1
    cuts = [0]
    while cuts[-1] < n:
        lo = cuts[-1]
        hi = min(n, lo + MAX_BATCH_RECORDS)
        limit = int(offsets[lo]) + MAX_BATCH_BYTES
        if int(offsets[hi]) > limit:
            hi = int(np.searchsorted(offsets, limit, side="right")) - 1
        if hi <= lo:
            if not oversize:
                raise FastaError("record longer than the batch size")
            hi = lo + 1
        cuts.append(hi)
    return cuts


def _pump(ctx: Context, arena: np.ndarray, offsets: np.ndarray, uniq: bool, want_bytes: bool = True, base_index: int = 0,
          threads: int = 0):
    """All batches of one piece of the input through the two slots of the C ABI (the bounded queue of parallel_fasta): the
    host packer (ck_pack2_host, `threads` threads) and the submit of batch b run while batch b - 1 is collected.
    canonicalize -> (canonical bytes of every record, compact; normalised lengths; None; None)
    uniq         -> (canonical bytes of the SURVIVORS only, compact -- the device compacts them, CK_F_SURVIVORS; lengths;
                     first_index of every record; indices of the survivors)"""
    from .core import pack2_host
    n = len(offsets) - 1
    cuts = _batches(offsets)
    lens = np.zeros(n, dtype=np.uint32)
    first = np.zeros(n, dtype=np.uint64) if uniq else None
    outs, keeps = [], []
    nb = len(cuts) - 1
    pend = {}
    for b in range(nb + 1):
        if b < nb:
            lo, hi = cuts[b], cuts[b + 1]
            rel = (offsets[lo: hi + 1] - offsets[lo]).astype(np.uint64)
            sub = arena[int(offsets[lo]): int(offsets[hi])]
            pb = pack2_host(sub, rel, normalize=True, threads=threads)
            if uniq:
                ctx.uniq_submit_packed(b & 1, pb, base_index + lo, no_bytes=not want_bytes, aligned=True, survivors=True)
            else:
                ctx.canon_submit_packed(b & 1, pb, aligned=True)
            pend[b] = pb                                       # keeps the pinned / host arrays alive until the wait
        if b >= 1:
            lo, hi = cuts[b - 1], cuts[b]
            pb = pend.pop(b - 1)
            if uniq:
                r = ctx.uniq_wait_survivors((b - 1) & 1, hi - lo, pb.total, want_bytes=want_bytes)
                first[lo:hi] = r["first"]
                lens[lo:hi] = r["lens"]
                idx = r["index"].astype(np.int64)
                keeps.append(idx + lo)
                if want_bytes and len(idx):
                    st = r["offsets"][:-1].astype(np.int64)
                    outs.append(r["bytes"][_region_mask(len(r["bytes"]), st, st + r["lens"][idx].astype(np.int64))])
            else:
                r = ctx.canon_wait((b - 1) & 1, hi - lo, pb.total, aligned=True)
                lens[lo:hi] = r["lens"]
                st = ctx.aligned_starts(pb.offsets).astype(np.int64)
                outs.append(r["out"][_region_mask(len(r["out"]), st, st + r["lens"].astype(np.int64))])
    body = np.concatenate(outs) if outs else np.zeros(0, dtype=np.uint8)
    keep = (np.concatenate(keeps) if keeps else np.zeros(0, dtype=np.int64)) if uniq else None
    return body, lens, first, keep


def _context(table_capacity: int) -> Context:
    return Context(max_batch_bytes=MAX_BATCH_BYTES, max_batch_records=MAX_BATCH_RECORDS, table_capacity=table_capacity)


def _piece_arena(recs: "Records"):
    seq_len = recs.seq_hi - recs.seq_lo
    offsets = np.zeros(len(recs) + 1, dtype=np.uint64)
    np.cumsum(seq_len, out=offsets[1:])
    return np.ascontiguousarray(recs.gather(recs.seq_lo, recs.seq_hi)), offsets, seq_len


def run_canonicalize(pieces, write, threads: int = 0) -> None:
    """`circkit canonicalize` over a stream of Records pieces (src/canonicalize.rs:7-51); `write(bytes)` gets the output"""
    ctx = None
    try:
        for recs in pieces:
            if len(recs) == 0:
                continue
            if ctx is None:
                ctx = _context(0)
            arena, offsets, _ = _piece_arena(recs)
            body, lens, _, _ = _pump(ctx, arena, offsets, False, threads=threads)
            heads = recs.gather(recs.head_lo, recs.head_hi)
            write(_assemble(heads, recs.head_hi - recs.head_lo, body, lens.astype(np.int64)))
    finally:
        if ctx is not None:
            ctx.close()


def _csv_field(f: bytes, delim: bytes) -> bytes:
    """csv 1.2.2 defaults (QuoteStyle::Necessary, double_quote, terminator '\\n')"""
    if any(c in f for c in (delim, b'"', b"\n", b"\r")):
        return b'"' + f.replace(b'"', b'""') + b'"'
    return f


def _check_ids(recs: "Records", which: np.ndarray) -> None:
    """record.id().unwrap() (src/uniq.rs:48,67): the id -- head up to the first ' ' -- must be UTF-8"""
    heads = recs.gather(recs.head_lo[which], recs.head_hi[which]).tobytes()
    try:
        heads.decode("utf-8")                                 # every head valid => every id valid (the common case)
        return
    except UnicodeDecodeError:
        pass
    for a, b in zip(recs.head_lo[which].tolist(), recs.head_hi[which].tolist()):
        recs.data[a:b].tobytes().split(b" ", 1)[0].decode("utf-8")


def run_uniq(pieces, write, canonical: bool = False, table_write=None, table_ext: str | None = None, table_capacity: int = 1 << 24,
             threads: int = 0) -> None:
    """`circkit uniq` over a stream of Records pieces (src/uniq.rs:15-88): one first-occurrence table on the device for the whole
    input, survivors written piece by piece in input order, duplicate rows to `table_write` as they are met."""
    ctx = None
    base = 0
    first_ids = {}                                             # global index of a first occurrence -> its id (for --table only)
    delim = b"\t" if table_ext == "tsv" else b","
    wrote_header = False
    try:
        for recs in pieces:
            n = len(recs)
            if n == 0:
                continue
            if ctx is None:
                ctx = _context(table_capacity)
            arena, offsets, seq_len = _piece_arena(recs)
            body, lens, first, keep_idx = _pump(ctx, arena, offsets, True, want_bytes=canonical, base_index=base, threads=threads)
            keep = np.zeros(n, dtype=bool)
            keep[keep_idx] = True                               # first occurrence in input order (src/uniq.rs:47-48)
            _check_ids(recs, np.ones(n, dtype=bool) if table_write is not None else keep)
            head_len = (recs.head_hi - recs.head_lo)[keep]
            heads = recs.gather(recs.head_lo[keep], recs.head_hi[keep])
            if canonical:                                       # src/uniq.rs:53-56: the device returned the survivors' bytes only
                bodies, body_len = body, lens.astype(np.int64)[keep]
            else:                                               # raw record.seq(), internal line breaks included (:57-59)
                bodies, body_len = recs.gather(recs.seq_lo[keep], recs.seq_hi[keep]), seq_len[keep]
            write(_assemble(heads, head_len, bodies, body_len))
            if table_write is not None:                         # src/uniq.rs:62-71, csv 1.2.2 defaults
                def rec_id(i):
                    return recs.data[recs.head_lo[i]: recs.head_hi[i]].tobytes().split(b" ", 1)[0]
                for i in keep_idx.tolist():
                    first_ids[base + i] = rec_id(i)
                rows = bytearray()
                for i in np.flatnonzero(~keep).tolist():
                    if not wrote_header:
                        rows += b"id" + delim + b"duplicate_id\n"
                        wrote_header = True
                    rows += _csv_field(first_ids[int(first[i])], delim) + delim + _csv_field(rec_id(i), delim) + b"\n"
                table_write(bytes(rows))
            base += n
    finally:
        if ctx is not None:
            ctx.close()


def canonicalize(fasta: bytes) -> bytes:
    """bytes of a FASTA file -> bytes `circkit canonicalize` writes (src/canonicalize.rs:7-51)"""
    out = []
    run_canonicalize(iter_records([fasta] if fasta else []), out.append)
    return b"".join(out)


def uniq(fasta: bytes, canonical: bool = False, table_ext: str | None = None):
    """bytes of a FASTA file -> (bytes `circkit uniq` writes, bytes of the --table file or None) (src/uniq.rs:15-88)"""
    out, table = [], ([] if table_ext is not None else None)
    n_upper = fasta.count(b">") + 1
    run_uniq(iter_records([fasta] if fasta else []), out.append, canonical, table.append if table is not None else None, table_ext,
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


def _pump_mono(ctx: Context, big: "Context | None", arena: np.ndarray, offsets: np.ndarray, opts):
    """All batches of one piece through the two slots (ck_mono_submit / ck_mono_wait): the submit of batch b runs while
    batch b - 1 is collected.  A record longer than MAX_BATCH_BYTES is a batch of its own on `big`, a context whose staging
    fits it.  -> (indices of the written records, increasing; their bytes, concatenated; monomer_len[n]; full_len[n])"""
    n = len(offsets) - 1
    cuts = _batches(offsets, oversize=True)
    mono_len = np.zeros(n, dtype=np.int64)
    full_len = np.zeros(n, dtype=np.int64)
    idxs, outs = [], []
    nb = len(cuts) - 1
    pend = {}
    for b in range(nb + 1):
        if b < nb:
            lo, hi = cuts[b], cuts[b + 1]
            rel = (offsets[lo: hi + 1] - offsets[lo]).astype(np.uint64)
            sub = arena[int(offsets[lo]): int(offsets[hi])]
            c = big if int(rel[-1]) > MAX_BATCH_BYTES else ctx
            c.mono_submit(b & 1, sub, rel, opts)
            pend[b] = (c, sub, rel)                              # keeps the host arrays alive until the wait
        if b >= 1:
            lo, hi = cuts[b - 1], cuts[b]
            c, _, rel = pend.pop(b - 1)
            r = c.mono_wait((b - 1) & 1, hi - lo, int(rel[-1]))
            mono_len[lo:hi] = r["monomer_len"]
            full_len[lo:hi] = r["full_len"]
            if r["n_written"]:
                idx = r["index"].astype(np.int64)
                st = r["offsets"][:-1].astype(np.int64)
                idxs.append(idx + lo)
                outs.append(r["bytes"][_region_mask(len(r["bytes"]), st, st + mono_len[lo + idx])])
    written = np.concatenate(idxs) if idxs else np.zeros(0, dtype=np.int64)
    body = np.concatenate(outs) if outs else np.zeros(0, dtype=np.uint8)
    return written, body, mono_len, full_len


def run_monomerize(pieces, write, opts, table_write=None, table_ext: str | None = None) -> None:
    """`circkit monomerize` over a stream of Records pieces (src/monomerize.rs:16-160): `opts` from mono_options; normalisation,
    the monomer search, the length / overlap filters of the consumer closure and the extraction of full_seq[..end] run on the
    device; `write(bytes)` gets the output ('>' head '\\n' monomer '\\n'), `table_write` the --table rows as pieces complete."""
    ctx = big = None
    delim = b"\t" if table_ext == "tsv" else b","
    wrote_header = False
    try:
        for recs in pieces:
            n = len(recs)
            if n == 0:
                continue
            arena, offsets, seq_len = _piece_arena(recs)
            longest = int(seq_len.max())
            if ctx is None:
                ctx = _context(0)
            if longest > MAX_BATCH_BYTES and (big is None or big.max_batch_bytes < longest):
                if big is not None:
                    big.close()
                big = Context(max_batch_bytes=longest, max_batch_records=1)
            written, body, mono_len, full_len = _pump_mono(ctx, big, arena, offsets, opts)
            heads = recs.gather(recs.head_lo[written], recs.head_hi[written])
            write(_assemble(heads, (recs.head_hi - recs.head_lo)[written], body, mono_len[written]))
            if table_write is not None and len(written):      # :145-154, csv 1.2.2 defaults: header with the first row
                rows = bytearray()
                if not wrote_header:
                    rows += delim.join([b"id", b"original_length", b"monomer_length"]) + b"\n"
                    wrote_header = True
                for i in written.tolist():
                    head = recs.data[recs.head_lo[i]: recs.head_hi[i]].tobytes()
                    head.decode("utf-8")                         # std::str::from_utf8(record.head()).unwrap()
                    rows += delim.join([_csv_field(head, delim), b"%d" % full_len[i], b"%d" % mono_len[i]]) + b"\n"
                table_write(bytes(rows))
    finally:
        for c in (ctx, big):
            if c is not None:
                c.close()


def monomerize(fasta: bytes, sensitive: bool = False, seed_length: int = 10, max_mismatch=None, min_identity=None,
               min_overlap=None, min_overlap_percent=None, min_length: int = 0, max_length=None, keep_all: bool = False,
               table_ext: str | None = None):
    """bytes of a FASTA file -> (bytes `circkit monomerize` writes, bytes of the --table file or None)
    (src/monomerize.rs:16-160), through run_monomerize"""
    opts = mono_options(sensitive, seed_length, max_mismatch, min_identity, min_overlap, min_overlap_percent, min_length,
                        max_length, keep_all)
    out, table = [], ([] if table_ext is not None else None)
    run_monomerize(iter_records([fasta] if fasta else []), out.append, opts, table.append if table is not None else None, table_ext)
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
        # every subcommand streams: decompress, split, (pack,) process and write piece by piece (src/utils.rs:9-72)
        pieces = iter_records(iter_input(args.input))
        first = next(pieces, None)                              # open the input (and fail on it) before the output is created

        def chain():
            if first is not None:
                yield first
            yield from pieces
        w = Writer(args.output)
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
                cap = 1 << 24
                if args.input is not None:
                    # distinct canonical forms the table must hold: bounded by the record count, itself bounded by the input size
                    # (a record needs >= 4 bytes; compressed DNA rarely beats 4x)
                    sz = os.path.getsize(args.input)
                    cap = max(1 << 16, min(1 << 30, sz if args.input.rsplit(".", 1)[-1] in ("gz", "bz2", "xz", "zst") else sz // 4))
                run_uniq(chain(), w.write, args.canonicalize, tf.write if tf else None, ext, table_capacity=cap, threads=threads)
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
