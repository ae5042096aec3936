"""The device bzip2 encoder (ck_bzip2_submit / ck_bzip2_wait) against libbz2: every stream it writes is byte for byte
bz2.compress(x, 9).  Sizes around the RLE1 block cut, runs across it, every table count, code lengths past 17, periodic
blocks on both of libbzip2's sort paths, a multi-block stream fed in calls of mixed sizes, and the CLI's `.bz2` output."""
import bz2
import os
import random
import shutil
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
FIX = os.path.join(HERE, "golden", "fixtures")
MAX = 64 << 20
BLOCK_MAX = 899981


@pytest.fixture(scope="module")
def ctx():
    from circkit_b200 import Context
    c = Context(max_batch_bytes=0, max_batch_records=0)
    yield c
    c.close()


def encode(ctx, data, sizes=None):
    """one bzip2 stream of `data`, fed in calls of `sizes` new bytes each (one call when None), the caller's framing"""
    from circkit_b200 import cli
    parts, tail, bits, nbits, crc, pos = [cli.BZIP2_HEADER], b"", 0, 0, 0, 0
    for n in sizes or []:
        buf = tail + data[pos:pos + n]
        pos += n
        if buf:
            out, consumed, bits, nbits, crc = ctx.bzip2(buf, False, bits, nbits, crc)
            parts.append(out)
            tail = buf[consumed:]
    buf = tail + data[pos:]
    if buf:
        out, consumed, bits, nbits, crc = ctx.bzip2(buf, True, bits, nbits, crc)
        assert consumed == len(buf)
        parts.append(out)
    v = (bits << 80 | cli.BZIP2_EOS << 32 | crc) << (-(nbits + 80) % 8)
    parts.append(v.to_bytes((nbits + 87) // 8, "big"))
    return b"".join(parts)


def check(ctx, data, sizes=None, decode=False):
    data = bytes(data)
    got = encode(ctx, data, sizes)
    want = bz2.compress(data, 9)
    if got != want:
        i = next((k for k in range(min(len(got), len(want))) if got[k] != want[k]), min(len(got), len(want)))
        raise AssertionError("%d input bytes: %d vs libbz2's %d bytes, first difference at byte %d"
                             % (len(data), len(got), len(want), i))
    if decode and shutil.which("bzip2"):
        assert subprocess.run(["bzip2", "-dc"], input=got, capture_output=True, check=True).stdout == data
    return got


def no_runs(rng, n):
    """n bytes with no two equal neighbours: every byte is one RLE1 byte"""
    return (np.cumsum(rng.integers(1, 256, n)) % 256).astype(np.uint8).tobytes()


def test_argument_and_state_errors(ctx):
    from circkit_b200.core import CircKitError
    with pytest.raises(CircKitError):
        ctx.bzip2_submit(0, b"", True)
    with pytest.raises(CircKitError):
        ctx.bzip2_submit(0, b"x", True, 0, 8, 0)
    with pytest.raises(CircKitError):
        ctx.bzip2_wait(1)
    ctx.bzip2_submit(1, b"abc", True)
    with pytest.raises(CircKitError):
        ctx.bzip2_submit(1, b"abc", True)
    ctx.bzip2_wait(1)
    check(ctx, b"abc")


def test_small_inputs_and_symbol_maps(ctx):
    check(ctx, b"x", decode=True)
    check(ctx, bytes(range(256)) * 5, decode=True)
    check(ctx, b"A" * 1000)
    check(ctx, b"AB" * 501 + b"A")
    check(ctx, b">a\n>a\n", decode=True)
    rng = random.Random(1)
    check(ctx, bytes(rng.randrange(256) for _ in range(30000)), decode=True)


@pytest.mark.parametrize("L", [3, 4, 5, 255, 256, 259, 510])
def test_runs(ctx, L):
    check(ctx, b"C" * L)
    check(ctx, b"xy" + b"C" * L + b"z" + b"C" * L)


@pytest.mark.parametrize("total", [BLOCK_MAX - 1, BLOCK_MAX, BLOCK_MAX + 1])
def test_rle1_lengths_at_the_block_cut(ctx, total):
    rng = np.random.default_rng(total)
    x = no_runs(rng, total)
    check(ctx, x)
    check(ctx, x + bytes([x[-1] ^ 1]) * 3)                # a run pending across the cut
    check(ctx, x + bytes([x[-1] ^ 1]) * 300)


def test_255_run_at_the_cut(ctx):
    rng = np.random.default_rng(7)
    x = no_runs(rng, BLOCK_MAX - 5)
    c = bytes([x[-1] ^ 1])
    for y in (x + c * 255, x + c * 255 + c * 10 + b"q", x + c * 254 + b"q" * 40, x + c * 600 + no_runs(rng, 1000)):
        check(ctx, y)
        check(ctx, y, sizes=[len(y) - 7])                 # the same stream with the last bytes in a final call


def test_table_counts_around_their_limits(ctx):
    rng = random.Random(9)
    for t in (200, 600, 1200, 2400):
        for n in range(t - 3, t + 3):
            check(ctx, bytes(rng.randrange(256) for _ in range(n)))


def test_code_lengths_past_17(ctx):
    fib = [1, 1]
    while len(fib) < 27:
        fib.append(fib[-1] + fib[-2])
    rng = random.Random(4)
    sym = [i for i, f in enumerate(fib) for _ in range(f)]
    rng.shuffle(sym)
    check(ctx, bytes(s * 7 % 256 for s in sym), decode=True)
    check(ctx, bytes(sym[:200000]))


def fasta(rng, nbytes, dup=0.3, rec=5000):
    recs, parts, size, i = [], [], 0, 0
    while size < nbytes:
        if recs and rng.random() < dup:
            body = rng.choice(recs[-50:])
        else:
            body = bytes(rng.choice(b"ACGT") for _ in range(rec))
            recs.append(body)
        r = b">r%d\n%s\n" % (i, body)
        parts.append(r)
        size += len(r)
        i += 1
    return b"".join(parts)


def test_fasta_with_copied_records(ctx):
    check(ctx, fasta(random.Random(2), 3 << 20), decode=True)


@pytest.mark.parametrize("k", [3, 1000, 3400, 20000, 100000])
def test_periodic_blocks(ctx, k):
    check(ctx, b">a\n" * k)
    check(ctx, b"AC" * k)


def test_periodic_900k_block(ctx):
    check(ctx, (b"ACGTTGCAx" * 100000)[:BLOCK_MAX])
    check(ctx, b">a\n" * 300000, decode=True)


def test_multi_block_stream_in_mixed_calls(ctx):
    rng = np.random.default_rng(11)
    rec = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, 40 << 20)]
    pieces, size = [], 0
    r = random.Random(12)
    while size < 200 << 20:
        if r.random() < 0.3 and size > 0:
            a = r.randrange(0, (40 << 20) - 6000)
            body = rec[a:a + 5000].tobytes()
        elif r.random() < 0.05:
            body = bytes([r.choice(b"ACGTN")]) * r.randint(4, 2000)
        else:
            a = r.randrange(0, (40 << 20) - 3000)
            body = rec[a:a + r.randint(200, 3000)].tobytes()
        pieces.append(b">s%d\n" % len(pieces) + body + b"\n")
        size += len(pieces[-1])
    data = b"".join(pieces)
    sizes, left = [], len(data) - 1000
    while left > 0:
        n = r.choice([1, 1, 7, 65536, 3 << 20, 17 << 20, 18 << 20])
        n = min(n, left)
        sizes.append(n)
        left -= n
    check(ctx, data, sizes=sizes, decode=True)


def _cli_bz2(tmp_path, argv, src, tag):
    """run argv on src with -o plain and -o .bz2; the .bz2 is bz2.compress of the plain output"""
    from circkit_b200 import cli
    plain, b2 = (str(tmp_path / ("%s%s" % (tag, s))) for s in (".fa", ".fa.bz2"))
    extra = lambda o: ["--table", o + ".tsv"] if "--table" in argv else []     # noqa: E731
    args = [a for a in argv if a != "--table"]
    for o in (plain, b2):
        assert cli.main(args[:1] + [src, "-o", o] + args[1:] + extra(o)) == 0
    p = open(plain, "rb").read()
    assert open(b2, "rb").read() == bz2.compress(p, 9)
    if "--table" in argv:
        assert open(b2 + ".tsv", "rb").read() == open(plain + ".tsv", "rb").read()
    return p


def test_cli_bz2_output_is_libbz2_of_the_plain_output(tmp_path, monkeypatch, capsys):
    from circkit_b200 import cli
    monkeypatch.setattr(cli, "MAX_BATCH_BYTES", 4096)      # many batches: many writes
    monkeypatch.setattr(cli, "MAX_BATCH_RECORDS", 16)
    rep = os.path.join(FIX, "repeated", "in.fasta")
    _cli_bz2(tmp_path, ["canonicalize"], rep, "c")
    _cli_bz2(tmp_path, ["uniq", "-c", "--table"], rep, "u")
    rng = random.Random(21)
    src = str(tmp_path / "in.fa")
    open(src, "wb").write(fasta(rng, 300000, rec=700))
    _cli_bz2(tmp_path, ["canonicalize"], src, "sc")
    _cli_bz2(tmp_path, ["uniq", "-c", "--table"], src, "su")
    mono = b"".join(b">m%d\n%s\n" % (i, (u * 3)[:len(u) * 2 + 7]) for i, u in
                    enumerate(bytes(rng.choice(b"ACGT") for _ in range(rng.randint(30, 200))) for _ in range(400)))
    msrc = str(tmp_path / "mono.fa")
    open(msrc, "wb").write(mono)
    _cli_bz2(tmp_path, ["monomerize"], msrc, "m")
    cap = capsys.readouterr()
    assert cap.out == "" and cap.err == ""
