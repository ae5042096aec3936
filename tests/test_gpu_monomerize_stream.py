"""`monomerize` through the two-slot batch API (ck_mono_submit / ck_mono_wait) and the streaming CLI driver
(cli.run_monomerize): byte for byte against the oracle's restatement of the driver over inputs cut into many pieces and
batches, records longer than a batch, `main` with compressed input and output, the library semantics of the batch API
without normalisation, a bench-shaped file of 1 M records, and the API's error codes."""
import gzip
import os
import random

import numpy as np
import pytest

from oracle import cli as ocli

pytestmark = pytest.mark.gpu

OPTION_SETS = [
    dict(), dict(sensitive=True), dict(seed_length=5, max_mismatch=2), dict(min_identity=0.9, keep_all=True, table_ext="csv"),
    dict(seed_length=12, min_identity=0.95, min_length=30, max_length=100, table_ext="tsv"),
    dict(min_overlap=20, min_overlap_percent=0.6, keep_all=True, table_ext="csv"), dict(seed_length=63, keep_all=True),
]


def _fasta(rng, n):
    """concatemers and noise; CRLF and LF, wrapped and unwrapped lines, ' ' / '\\t' inside lines, empty records, missing
    final newlines"""
    recs = []
    for i in range(n):
        unit = bytes(rng.choice(b"ACGT") for _ in range(rng.randint(8, 120)))
        kind = rng.randrange(6)
        if kind == 0:
            s = unit * rng.randint(2, 3)
        elif kind == 1:
            s = unit * 2 + unit[: rng.randint(0, len(unit))]
        elif kind == 2:
            s = bytearray(unit * 2)
            s[rng.randrange(len(s))] = rng.choice(b"ACGTN")
            s = bytes(s)
        elif kind == 3:
            s = bytes(rng.choice(b"ACGTacgtnNRYu") for _ in range(rng.randint(0, 200)))
        elif kind == 4:
            s = b""
        else:
            s = bytearray(unit * 2)
            for _ in range(rng.randint(1, 3)):
                s.insert(rng.randrange(len(s) + 1), rng.choice(b" \t\r"))
            s = bytes(s)
        width = rng.choice([0, 7, 60])
        eol = rng.choice([b"\n", b"\r\n"])
        body = s if not width else eol.join(s[k: k + width] for k in range(0, len(s), width))
        recs.append(b">r%d some, \"text\"" % i + eol + body + (eol if body or rng.random() < 0.5 else b""))
    data = b"".join(recs)
    return data if data.endswith(b"\n") or rng.random() < 0.5 else data[:-1]


def _run(cli, data, kw, chunk):
    from circkit_b200.cli import iter_records
    kw = dict(kw)
    ext = kw.pop("table_ext", None)
    out, table = [], []
    pieces = [data[k: k + chunk] for k in range(0, len(data), chunk)]
    cli.run_monomerize(iter_records(pieces), out.append, cli.mono_options(**kw), table.append if ext else None, ext)
    return b"".join(out), (b"".join(table) if ext else None)


@pytest.fixture
def small_batches(monkeypatch):
    from circkit_b200 import cli
    monkeypatch.setattr(cli, "MAX_BATCH_BYTES", 2048)
    monkeypatch.setattr(cli, "MAX_BATCH_RECORDS", 7)
    return cli


@pytest.mark.parametrize("kw", OPTION_SETS)
def test_pieces_and_batches_match_the_oracle_driver(small_batches, kw):
    cli = small_batches
    rng = random.Random(len(repr(kw)) + 17)
    data = _fasta(rng, 300)
    assert _run(cli, data, kw, 3000) == ocli.cli_monomerize(data, **kw)


def test_empty_records_and_batches_with_nothing_written(small_batches):
    cli = small_batches
    data = b"".join(b">e%d\n\n" % i for i in range(20)) + b">x\nACGTACGTAC\n" + b"".join(b">f%d\n" % i for i in range(20))
    for kw in (dict(keep_all=True, table_ext="csv"), dict(table_ext="tsv")):
        assert _run(cli, data, kw, 64) == ocli.cli_monomerize(data, **kw)
    assert _run(cli, data, dict(table_ext="tsv"), 64) == (b"", b"")


def test_record_longer_than_a_batch(small_batches):
    cli = small_batches
    rng = random.Random(3)
    unit = bytes(rng.choice(b"ACGT") for _ in range(1500))
    long_rec = unit * 3 + unit[:700]                           # 5200 bytes > MAX_BATCH_BYTES = 2048
    # CRLF lines of 511 / 1023 bases: a '\r' at byte 511 of a 512-byte step, whose '\n' only the next step holds (the look-ahead
    # of the warp's last lane)
    unit2 = bytes(rng.choice(b"ACGT") for _ in range(700))
    crlf = unit2 * 2 + unit2[:200]
    plain = bytes(rng.choice(b"ACGT") for _ in range(1600))     # no monomer: -k writes all of full_seq
    data = (b">a\nACGTACGTACGTAAAA\n>long one\n" + b"\n".join(long_rec[k: k + 70] for k in range(0, len(long_rec), 70))
            + b"\n>b\n" + unit[:40] * 2 + b"\n>long two\r\n" + long_rec * 2 + b"\r\n"
            + b">crlf 511\r\n" + b"\r\n".join(crlf[k: k + 511] for k in range(0, len(crlf), 511)) + b"\r\n"
            + b">crlf 1023\r\n" + b"\r\n".join(long_rec[k: k + 1023] for k in range(0, len(long_rec), 1023)) + b"\r\n"
            + b">crlf whole\r\n" + b"\r\n".join(plain[k: k + 511] for k in range(0, len(plain), 511)) + b"\r\n")
    for kw in (dict(table_ext="csv"), dict(keep_all=True, seed_length=20)):
        assert _run(cli, data, kw, 1000) == ocli.cli_monomerize(data, **kw)


def test_main_gz_in_zst_out_with_table(tmp_path, monkeypatch, small_batches):
    cli = small_batches
    data = _fasta(random.Random(5), 400)
    src = tmp_path / "in.fa.gz"
    src.write_bytes(gzip.compress(data))
    dst, tab = tmp_path / "out.fa.zst", tmp_path / "x.tsv"
    orig = cli.iter_input
    monkeypatch.setattr(cli, "iter_input", lambda p: orig(p, chunk_bytes=4096))
    assert cli.main(["monomerize", str(src), "-o", str(dst), "--table", str(tab), "-k", "--seed-length", "8"]) == 0
    want_out, want_tab = cli.monomerize(data, seed_length=8, keep_all=True, table_ext="tsv")
    assert cli.read_input(str(dst)) == want_out
    assert tab.read_bytes() == want_tab
    assert want_tab.count(b"id\toriginal_length\tmonomer_length") == 1
    assert (want_out, want_tab) == ocli.cli_monomerize(data, seed_length=8, keep_all=True, table_ext="tsv")


@pytest.mark.parametrize("mode", ["plain", "sensitive", "first_only"])
def test_batch_api_without_normalisation_is_the_library(mode):
    from circkit_b200 import _native as N
    from circkit_b200.core import Context
    from circkit_b200.monomerize import Monomerizer
    rng = random.Random(11)
    seqs = []
    for _ in range(500):
        unit = bytes(rng.choice(b"ACGTN") for _ in range(rng.randint(5, 90)))
        seqs.append((unit * rng.randint(1, 4))[: rng.randint(0, 400)])
    seqs += [b"", b"acgtACGT\n\r acgtACGT", b"A" * 64]
    off = np.zeros(len(seqs) + 1, dtype=np.uint64)
    np.cumsum([len(s) for s in seqs], out=off[1:])
    arena = np.frombuffer(b"".join(seqs), dtype=np.uint8).copy()
    flags = {"plain": 0, "sensitive": N.CK_MONO_SENSITIVE, "first_only": N.CK_MONO_FIRST_ONLY}[mode]
    opts = N.CkMonoOptions(7, flags | N.CK_MONO_KEEP_ALL, 0, 0.9, 0, 2**64 - 1, 0, float("nan"))
    ctx = Context(max_batch_bytes=1 << 20, max_batch_records=1 << 12)
    try:
        ctx.mono_submit(1, arena, off, opts, normalize=False)
        r = ctx.mono_wait(1, len(seqs), int(off[-1]))
    finally:
        ctx.close()
    m = Monomerizer(7, overlap_min_identity=0.9)
    want = m.end_indices(seqs, sensitive=mode == "sensitive", first_only=mode == "first_only")
    got = [None if v == N.CK_MONO_NONE else int(v) for v in r["end"].tolist()]
    assert got == want
    assert r["n_written"] == len(seqs) and r["index"].tolist() == list(range(len(seqs)))
    assert r["full_len"].tolist() == [len(s) for s in seqs]
    for k, s in enumerate(seqs):
        e = len(s) if want[k] is None else want[k]
        o = int(r["offsets"][k])
        assert o % 16 == 0 and int(r["monomer_len"][k]) == e
        assert r["bytes"][o: o + e].tobytes() == s[:e], k


def test_bench_shaped_file_against_the_compiled_port(tmp_path):
    """1 M single-line ACGT concatemers (2.3 copies of a 250-400 nt unit, 1 % substitutions), `-k --table`, no filters: every
    monomer_length equals the compiled oracle port's end index, or the whole record where the port finds none, and the output
    holds exactly those prefixes of the records (records of 575-920 bytes: the gather carries its stage across steps)"""
    from circkit_b200 import cli
    from oracle.monomerize import c_end_indices_batch
    n = 1_000_000
    rng = np.random.default_rng(1)
    unit = rng.integers(250, 401, n)
    rec_len = (unit * 2.3).astype(np.int64)
    off = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(rec_len, out=off[1:])
    arena = np.empty(int(off[-1]), dtype=np.uint8)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    for lo in range(0, n, 100_000):                            # bench.py's hash of (record, position mod unit), in blocks
        hi = min(n, lo + 100_000)
        rec = np.repeat(np.arange(lo, hi, dtype=np.int64), rec_len[lo:hi])
        pos = np.arange(int(off[lo]), int(off[hi]), dtype=np.int64) - off[rec]
        h = ((rec * 1000003 + pos % unit[rec]) * 2654435761) % 4294967296
        a = acgt[((h >> 13) ^ (h >> 7)) & 3]
        mut = rng.random(len(a)) < 0.01
        a[mut] = acgt[rng.integers(0, 4, int(mut.sum()))]
        arena[int(off[lo]): int(off[hi])] = a
    want = c_end_indices_batch(arena, off.astype(np.uint64), 10, overlap_min_identity=0.95, threads=os.cpu_count() or 1)
    path = tmp_path / "bench.fa"
    with open(path, "wb") as f:
        for lo in range(0, n, 100_000):
            hi = min(n, lo + 100_000)
            heads = [b">m%d\n" % i for i in range(lo, hi)]
            f.write(b"".join(h_ + arena[off[i]: off[i + 1]].tobytes() + b"\n" for h_, i in zip(heads, range(lo, hi))))
    out, table = [], []
    cli.run_monomerize(cli.iter_records(cli.iter_input(str(path))), out.append,
                       cli.mono_options(seed_length=10, min_identity=0.95, keep_all=True), table.append, "tsv")
    rows = b"".join(table).split(b"\n")
    assert rows[0] == b"id\toriginal_length\tmonomer_length" and rows[-1] == b"" and len(rows) == n + 2
    got = np.array([int(r.rsplit(b"\t", 1)[1]) for r in rows[1:-1]], dtype=np.int64)
    full = np.array([int(r.split(b"\t")[1]) for r in rows[1:-1]], dtype=np.int64)
    assert np.array_equal(full, rec_len)
    end = np.where(want == 0xFFFFFFFF, rec_len, want.astype(np.int64))
    assert np.array_equal(got, end)
    assert (want != 0xFFFFFFFF).mean() > 0.5
    ab = arena.tobytes()
    assert b"".join(out) == b"".join(b">m%d\n" % i + ab[o: o + e] + b"\n" for i, (o, e) in enumerate(zip(off[:-1].tolist(), end.tolist())))


def test_record_beyond_2_30_bytes():
    """the batch API's record limit is the path's 32-bit lengths, not canonicalize's 2^30 symbols: one record of 2^30 + 128
    bytes (two copies of a random 2^29 + 64-byte unit) through normalisation, the monomer search, the filters and the gather"""
    from circkit_b200 import _native as N
    from circkit_b200.core import Context
    L = (1 << 29) + 64
    unit = np.frombuffer(b"ACGT", dtype=np.uint8)[np.random.default_rng(5).integers(0, 4, L, dtype=np.uint8)]
    arena = np.concatenate([unit, unit])
    off = np.array([0, 2 * L], dtype=np.uint64)
    assert 2 * L > 1 << 30
    opts = N.CkMonoOptions(32, 0, 0, -1.0, 0, 2**64 - 1, 0, float("nan"))
    ctx = Context(max_batch_bytes=2 * L, max_batch_records=1)
    try:
        ctx.mono_submit(0, arena, off, opts)
        r = ctx.mono_wait(0, 1, 2 * L)
    finally:
        ctx.close()
    assert int(r["end"][0]) == L and int(r["full_len"][0]) == 2 * L and int(r["monomer_len"][0]) == L
    assert r["n_written"] == 1 and int(r["offsets"][1]) == L
    assert np.array_equal(r["bytes"][:L], unit)


def test_batch_api_errors():
    from circkit_b200 import _native as N
    from circkit_b200.core import CircKitError, Context
    ctx = Context(max_batch_bytes=1 << 16, max_batch_records=64)
    arena = np.frombuffer(b"ACGTACGTACGTACGTACGT", dtype=np.uint8).copy()
    off = np.array([0, 20], dtype=np.uint64)
    good = N.CkMonoOptions(4, 0, 0, -1.0, 0, 2**64 - 1, 0, float("nan"))
    try:
        with pytest.raises(CircKitError) as e:
            ctx.mono_wait(0, 1, 20)
        assert e.value.code == N.CK_ERR_STATE
        ctx.mono_submit(0, arena, off, good)
        with pytest.raises(CircKitError) as e:
            ctx.mono_submit(0, arena, off, good)
        assert e.value.code == N.CK_ERR_STATE
        with pytest.raises(CircKitError) as e:                # a mono batch is not collected by the uniq / canon waits
            ctx.canon_wait(0, 1, 20)
        assert e.value.code == N.CK_ERR_STATE
        ctx.canon_submit(1, arena, off, normalize=True)        # the other slot takes a canonicalize batch meanwhile
        r = ctx.mono_wait(0, 1, 20)
        assert r["n_written"] == 1 and r["bytes"][:4].tobytes() == b"ACGT" and int(r["monomer_len"][0]) == 4
        ctx.canon_wait(1, 1, 20)
        for bad in (N.CkMonoOptions(0, 0, 0, -1.0, 0, 2**64 - 1, 0, float("nan")),
                    N.CkMonoOptions(64, 0, 0, -1.0, 0, 2**64 - 1, 0, float("nan")),
                    N.CkMonoOptions(4, 0, 3, 0.9, 0, 2**64 - 1, 0, float("nan"))):
            with pytest.raises(CircKitError) as e:
                ctx.mono_submit(0, arena, off, bad)
            assert e.value.code == N.CK_ERR_ARG
        ctx.mono_submit(0, arena, off, good)                   # the slot is usable after the refusals
        assert ctx.mono_wait(0, 1, 20)["n_written"] == 1
    finally:
        ctx.close()
