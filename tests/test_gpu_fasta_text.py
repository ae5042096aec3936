"""The FASTA text batch API (ck_fasta_submit / ck_fasta_wait): the device's record split against cli.Records on adversarial
texts, the framed output of every command byte for byte against the oracle's restatement of the CLI (reference fixtures,
a 20 k-record synthetic file, the monomerize option sets, many tiny batches on alternating slots with the uniq table
spanning them), a text batch beside a host-buffer batch on the other slot, the error codes, and `main` end to end."""
import os
import random

import numpy as np
import pytest

import oracle
from oracle import cli as ocli

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
FIX = os.path.join(HERE, "golden", "fixtures")
GOLD = os.path.join(HERE, "golden", "oracle_cli")
MONO_FIX = os.path.join(HERE, "golden", "monomerize_fixtures")
FIXTURES = sorted(d for d in os.listdir(FIX) if os.path.isfile(os.path.join(FIX, d, "in.fasta")))
OPTION_SETS = [
    dict(), dict(sensitive=True), dict(seed_length=5, max_mismatch=2), dict(min_identity=0.9, keep_all=True, table_ext="csv"),
    dict(seed_length=12, min_identity=0.95, min_length=30, max_length=100, table_ext="tsv"),
    dict(min_overlap=20, min_overlap_percent=0.6, keep_all=True, table_ext="csv"), dict(seed_length=63, keep_all=True),
]

ADVERSARIAL = [
    b">a\r\nAC\r\nGT\r\n>b\r\n\r\n>c\r\nA C\tG\r\n",                 # CRLF, an empty record, whitespace inside a line
    b">only header",                                              # header only, no line break
    b">h1\n>h2\n>h3\nACGT",                                       # header-only records, last record without a final '\n'
    b">x\nAC>GT\nA>\n>y\n>z\nTT\n\n",                             # '>' inside sequence lines, a trailing empty line
    b">\n\n>\nA\n>",                                              # empty heads, a last record of '>' alone
    b">\xc3\xa9t\xe9 d\xff\nACGU\n>b \x80\r\nacgtn\r\n",          # non-ASCII (and non-UTF-8) headers
    b">r\r\r\nAC\r\r\n>s\rx\nA\r",                                 # '\r' trimmed once only; a bare '\r' inside a head
    b">" + b"long header " * 30 + b"\n" + b"ACGT" * 300 + b"\n>t\n" + b"\n".join([b"ACGTN" * 14] * 40),
]


def _ctx(**kw):
    from circkit_b200.core import Context
    return Context(**{"max_batch_bytes": 1 << 20, "max_batch_records": 1 << 12, **kw})


def _synthetic(n=20000, seed=17):
    """shaped like test_gpu_cli's synthetic file: wrapped lines, CRLF, lower case, RNA, IUPAC, rotated / reverse-complement
    duplicates"""
    rng = random.Random(seed)
    recs, lines = [], []
    for i in range(n):
        if recs and rng.random() < 0.3:
            s = rng.choice(recs)
            r = rng.randrange(len(s))
            s = s[r:] + s[:r]
            if rng.random() < 0.5:
                s = oracle.revcomp(s)
        else:
            s = bytes(rng.choice(b"ACGT") for _ in range(rng.randint(1, 600)))
            recs.append(s)
        if rng.random() < 0.1:
            s = s.lower()
        if rng.random() < 0.05:
            s = s.replace(b"T", b"U")
        if rng.random() < 0.05:
            k = rng.randrange(len(s))
            s = s[:k] + rng.choice([b"N", b"R", b"y", b"-", b"."]) + s[k + 1:]
        eol = b"\r\n" if rng.random() < 0.1 else b"\n"
        w = rng.choice([0, 60, 70])
        body = eol.join(s[k:k + w] for k in range(0, len(s), w)) if w else s
        lines.append(b">r%d some description" % i + eol + body + eol)
    return b"".join(lines)


def test_device_ranges_equal_the_host_split():
    from circkit_b200 import cli
    ctx = _ctx(table_capacity=1 << 12)
    try:
        for k, text in enumerate(ADVERSARIAL + [_synthetic(300, 3)]):
            recs = cli.Records(text)
            slot = k & 1
            for command in ("canonicalize", "uniq", "monomerize"):
                kw = dict(mono=cli.mono_options(keep_all=True)) if command == "monomerize" else {}
                n = ctx.fasta_submit(slot, text, command, **kw)
                r = ctx.fasta_wait(slot)
                assert n == len(recs), (k, command)
                assert r["head"][:, 0].tolist() == recs.head_lo.tolist(), (k, command)
                assert r["head"][:, 1].tolist() == recs.head_hi.tolist(), (k, command)
                if command == "monomerize":
                    assert r["full_len"].tolist() == [len(ocli.full_seq(recs.data[a:b].tobytes()))
                                                      for a, b in zip(recs.seq_lo.tolist(), recs.seq_hi.tolist())]
            ctx.uniq_reset()
            assert ctx.fasta_submit(slot, text, "canonicalize") == len(recs)
            assert ctx.fasta_wait(slot)["fasta"] == ocli.cli_canonicalize(text)
    finally:
        ctx.close()


def _api_run(ctx, text, command, canonical=False, mono=None, slot=0):
    n = ctx.fasta_submit(slot, text, command, canonical_body=canonical, mono=mono)
    r = ctx.fasta_wait(slot)
    assert len(r["head"]) == n
    return r


@pytest.mark.parametrize("d", FIXTURES)
def test_fixtures_through_the_api(d):
    data = open(os.path.join(FIX, d, "in.fasta"), "rb").read()
    gold = lambda name: open(os.path.join(GOLD, d + name), "rb").read()    # noqa: E731
    from circkit_b200 import cli
    text = cli._piece_text(data)                                    # the caller strips the leading blank lines
    ctx = _ctx(table_capacity=1 << 12)
    try:
        assert _api_run(ctx, text, "canonicalize")["fasta"] == gold(".canonicalize.out")
        r = _api_run(ctx, text, "uniq", slot=1)
        assert r["fasta"] == gold(".uniq.out")
        assert r["index"].tolist() == [i for i, f in enumerate(r["first"].tolist()) if f == i]
        ctx.uniq_reset()
        assert _api_run(ctx, text, "uniq", canonical=True)["fasta"] == gold(".uniq_c.out")
    finally:
        ctx.close()


@pytest.mark.parametrize("d", sorted(os.listdir(MONO_FIX)))
def test_monomerize_fixtures_through_the_api(d):
    from circkit_b200 import cli
    kw = {"min_overlap": dict(min_overlap=81), "min_overlap_percent_0.51": dict(min_overlap_percent=0.51),
          "min_overlap_percent_1.0": dict(min_overlap_percent=1.0), "min_overlap_percent_1.5": dict(min_overlap_percent=1.5)}[d]
    data = open(os.path.join(MONO_FIX, d, "in.fasta"), "rb").read()
    ctx = _ctx()
    try:
        r = _api_run(ctx, cli._piece_text(data), "monomerize", mono=cli.mono_options(**kw))
    finally:
        ctx.close()
    assert r["fasta"] == ocli.cli_monomerize(data, **kw)[0]
    want = {x.id: ocli.full_seq(x.seq) for x in ocli.parse_fasta(open(os.path.join(MONO_FIX, d, "out.fasta"), "rb").read())}
    assert {x.id: ocli.full_seq(x.seq) for x in ocli.parse_fasta(r["fasta"])} == want


def test_synthetic_file_through_the_cli():
    from circkit_b200 import cli
    data = _synthetic()
    assert cli.canonicalize(data) == ocli.cli_canonicalize(data, threads=4)
    for canon in (False, True):
        assert cli.uniq(data, canonical=canon, table_ext="csv") == ocli.cli_uniq(data, canonicalize=canon, table_ext="csv", threads=4)
    assert cli.monomerize(data, keep_all=True, table_ext="tsv") == ocli.cli_monomerize(data, keep_all=True, table_ext="tsv")


@pytest.fixture
def tiny_batches(monkeypatch):
    from circkit_b200 import cli
    monkeypatch.setattr(cli, "MAX_BATCH_BYTES", 700)
    monkeypatch.setattr(cli, "MAX_BATCH_RECORDS", 5)
    return cli


def _pieces(data, chunk):
    return [data[k: k + chunk] for k in range(0, len(data), chunk)]


@pytest.mark.parametrize("chunk", [97, 1500])
def test_tiny_batches_on_alternating_slots(tiny_batches, chunk):
    """many batches per piece and records straddling pieces: the uniq table spans the batches with the right base_index"""
    cli = tiny_batches
    rng = random.Random(chunk)
    # short records only (the batch size is 700 bytes), with many duplicates across batches
    recs = [r for r in (b">" + x.rstrip(b"\n") for x in _synthetic(400, chunk)[1:].split(b"\n>")) if len(r) < 600]
    data = b"\n".join(rng.choice(recs) for _ in range(600)) + b"\n"
    for command in ("canonicalize", "uniq"):
        out, table = [], []
        if command == "canonicalize":
            cli.run_canonicalize(cli.iter_text(_pieces(data, chunk)), out.append)
            assert b"".join(out) == ocli.cli_canonicalize(data)
        else:
            for canon in (False, True):
                out, table = [], []
                cli.run_uniq(cli.iter_text(_pieces(data, chunk)), out.append, canon, table.append, "csv", table_capacity=1 << 12)
                assert (b"".join(out), b"".join(table)) == ocli.cli_uniq(data, canonicalize=canon, table_ext="csv")
    for kw in OPTION_SETS:
        kw = dict(kw)
        ext = kw.pop("table_ext", None)
        out, table = [], []
        cli.run_monomerize(cli.iter_text(_pieces(data, chunk)), out.append, cli.mono_options(**kw), table.append if ext else None, ext)
        assert (b"".join(out), b"".join(table) if ext else None) == ocli.cli_monomerize(data, table_ext=ext, **kw)


def test_a_text_batch_beside_host_buffer_batches():
    from circkit_b200 import cli
    text = _synthetic(2000, 9)
    recs = cli.Records(text)
    seq = [recs.data[a:b].tobytes() for a, b in zip(recs.seq_lo.tolist(), recs.seq_hi.tolist())]
    off = np.zeros(len(seq) + 1, dtype=np.uint64)
    np.cumsum([len(s) for s in seq], out=off[1:])
    arena = np.frombuffer(b"".join(seq), dtype=np.uint8).copy()
    opts = cli.mono_options(keep_all=True)
    ctx = _ctx(table_capacity=1 << 14)
    try:
        # a monomerize text batch on slot 0 while a uniq host batch is on slot 1, then the other way round
        n = ctx.fasta_submit(0, text, "monomerize", mono=opts)
        ctx.uniq_submit(1, arena, off, 0, normalize=True)
        r = ctx.fasta_wait(0)
        u = ctx.uniq_wait(1, n, int(off[-1]))
        assert r["fasta"] == ocli.cli_monomerize(text, keep_all=True)[0]
        # the table now holds the batch: a uniq text batch of the same records at base_index n finds every first occurrence
        ctx.mono_submit(1, arena, off, opts)
        assert ctx.fasta_submit(0, text, "uniq", base_index=n) == n
        m = ctx.mono_wait(1, n, int(off[-1]))
        r2 = ctx.fasta_wait(0)
        assert r2["n_written"] == 0 and r2["fasta"] == b""
        assert np.array_equal(r2["first"], u["first"])
        assert m["n_written"] == n
    finally:
        ctx.close()


def test_error_codes():
    from circkit_b200 import _native as N
    from circkit_b200 import cli
    from circkit_b200.core import CircKitError, Context
    ctx = Context(max_batch_bytes=4096, max_batch_records=8)
    many = b"".join(b">r%d\nACGT\n" % i for i in range(9))                 # 9 records > max_batch_records
    good = b">a\nACGTACGTAC\n>b\nGGTT\n"

    def code(fn, *a, **kw):
        with pytest.raises(CircKitError) as e:
            fn(*a, **kw)
        return e.value.code
    try:
        assert code(ctx.fasta_submit, 0, b"ACGT\n>a\n", "canonicalize") == N.CK_ERR_ARG      # must begin with '>'
        assert code(ctx.fasta_submit, 0, b"\n>a\nAC\n", "canonicalize") == N.CK_ERR_ARG
        assert code(ctx.fasta_submit, 0, b">" + b"A" * 4096, "canonicalize") == N.CK_ERR_ARG  # > max_batch_bytes
        assert code(ctx.fasta_submit, 0, good, "uniq") == N.CK_ERR_STATE                     # table_capacity 0
        assert code(ctx.fasta_submit, 0, good, "monomerize") == N.CK_ERR_ARG                 # no options
        bad = N.CkMonoOptions(4, 0, 3, 0.9, 0, 2**64 - 1, 0, float("nan"))
        assert code(ctx.fasta_submit, 0, good, "monomerize", mono=bad) == N.CK_ERR_ARG
        assert code(ctx.fasta_submit, 1, many, "canonicalize") == N.CK_ERR_ARG             # more records than the slot takes
        assert ctx.fasta_submit(1, good, "canonicalize") == 2                               # ... and the slot stays usable
        assert code(ctx.fasta_submit, 1, good, "canonicalize") == N.CK_ERR_STATE            # busy
        assert code(ctx.canon_wait, 1, 2, 14) == N.CK_ERR_STATE                             # not collected by the other waits
        assert code(ctx.mono_wait, 1, 2, 14) == N.CK_ERR_STATE
        assert ctx.fasta_wait(1)["fasta"] == ocli.cli_canonicalize(good)
        assert code(ctx.fasta_wait, 1) == N.CK_ERR_STATE                                   # nothing left on the slot
        assert ctx.fasta_submit(0, b"", "canonicalize") == 0
        assert ctx.fasta_wait(0)["fasta"] == b""
    finally:
        ctx.close()
    big = Context(max_batch_bytes=(1 << 30) + 64, max_batch_records=1, table_capacity=16)
    try:
        text = np.full((1 << 30) + 5, ord("A"), dtype=np.uint8)
        text[:3] = np.frombuffer(b">a\n", dtype=np.uint8)
        assert code(big.fasta_submit, 0, text, "canonicalize") == N.CK_ERR_TOO_LONG        # 2^30 + 2 symbols
        assert code(big.fasta_submit, 0, text, "uniq") == N.CK_ERR_TOO_LONG
        assert big.fasta_submit(0, text[:(1 << 20)], "canonicalize") == 1
        assert len(big.fasta_wait(0)["fasta"]) == (1 << 20) + 1
    finally:
        big.close()
    peer = Context(max_batch_bytes=1 << 16, max_batch_records=16, table_capacity=16)
    try:
        peer.peer_attach([peer.peer_export(1, 0, 16)])                   # a peer group of one
        assert code(peer.fasta_submit, 0, good, "uniq") == N.CK_ERR_STATE
        assert peer.fasta_submit(0, good, "monomerize", mono=cli.mono_options()) == 2   # other commands still run
        peer.fasta_wait(0)
    finally:
        peer.close()


def test_main_non_utf8_id_in_uniq(tmp_path, capsys):
    from circkit_b200 import cli
    src = tmp_path / "in.fa"
    src.write_bytes(b">ok\nACGT\n>bad\xff id\nGGGG\n")
    assert cli.main(["uniq", str(src), "-o", str(tmp_path / "out.fa")]) == 1
    assert capsys.readouterr().err.startswith("Error:")
    src.write_bytes(b">ok\nACGT\n>dup\xff\nACGT\n")                       # a duplicate's id matters with --table only
    assert cli.main(["uniq", str(src), "-o", str(tmp_path / "out.fa")]) == 0
    assert (tmp_path / "out.fa").read_bytes() == b">ok\nACGT\n"
    assert cli.main(["uniq", str(src), "-o", str(tmp_path / "out.fa"), "--table", str(tmp_path / "t.csv")]) == 1
    assert capsys.readouterr().err.startswith("Error:")


def test_bench_shaped_file_through_main(tmp_path):
    """1 M single-line ACGT concatemers (bench.py's mono workload, as test_gpu_monomerize_stream builds it) through `main`
    with -k and --table: the table and the whole output against the compiled oracle port"""
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
    for lo in range(0, n, 100_000):
        hi = min(n, lo + 100_000)
        rec = np.repeat(np.arange(lo, hi, dtype=np.int64), rec_len[lo:hi])
        pos = np.arange(int(off[lo]), int(off[hi]), dtype=np.int64) - off[rec]
        h = ((rec * 1000003 + pos % unit[rec]) * 2654435761) % 4294967296
        a = acgt[((h >> 13) ^ (h >> 7)) & 3]
        mut = rng.random(len(a)) < 0.01
        a[mut] = acgt[rng.integers(0, 4, int(mut.sum()))]
        arena[int(off[lo]): int(off[hi])] = a
    want = c_end_indices_batch(arena, off.astype(np.uint64), 10, overlap_min_identity=0.95, threads=os.cpu_count() or 1)
    end = np.where(want == 0xFFFFFFFF, rec_len, want.astype(np.int64))
    ab = arena.tobytes()
    path = tmp_path / "bench.fa"
    with open(path, "wb") as f:
        f.write(b"".join(b">m%d\n" % i + ab[o: o + L] + b"\n" for i, (o, L) in enumerate(zip(off[:-1].tolist(), rec_len.tolist()))))
    out, tab = tmp_path / "out.fa", tmp_path / "t.tsv"
    assert cli.main(["monomerize", str(path), "-o", str(out), "-k", "--min-identity", "0.95", "--table", str(tab)]) == 0
    assert out.read_bytes() == b"".join(b">m%d\n" % i + ab[o: o + e] + b"\n" for i, (o, e) in enumerate(zip(off[:-1].tolist(), end.tolist())))
    rows = tab.read_bytes().split(b"\n")
    assert rows[0] == b"id\toriginal_length\tmonomer_length" and len(rows) == n + 2
    assert rows[1:-1] == [b"m%d\t%d\t%d" % (i, L, e) for i, (L, e) in enumerate(zip(rec_len.tolist(), end.tolist()))]
