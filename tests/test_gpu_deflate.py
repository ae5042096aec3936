"""The device DEFLATE encoder (ck_deflate_submit / ck_deflate_wait) against zlib: every fragment decodes alone with its
dictionary, has no final block, ends in a sync flush and carries the right CRC-32; sizes around the segment and block
limits, match distances at the window's edge, matches into the dictionary; and the CLI's `.gz` output through it."""
import gzip
import os
import random
import shutil
import subprocess
import zlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
FIX = os.path.join(HERE, "golden", "fixtures")
GOLD = os.path.join(HERE, "golden", "oracle_cli")
SEG = 65536
MAX = 64 << 20


@pytest.fixture(scope="module")
def ctx():
    from circkit_b200 import Context
    c = Context(max_batch_bytes=0, max_batch_records=0)
    yield c
    c.close()


def _zlib_raw(data, level):
    c = zlib.compressobj(level, zlib.DEFLATED, -15)
    return c.compress(data) + c.flush(zlib.Z_SYNC_FLUSH)


def check(ctx, data, dict=b"", crc=0):
    out, c = ctx.deflate(data, dict, crc)
    assert out.endswith(b"\x00\x00\xff\xff")
    d = zlib.decompressobj(-15, zdict=dict) if dict else zlib.decompressobj(-15)
    assert d.decompress(out) == data
    assert not d.eof and d.unused_data == b""            # no final block
    assert c == zlib.crc32(data, crc)
    assert len(out) <= ctx.deflate_bound(len(data))
    if len(data) >= 1 << 20:
        assert len(out) <= len(_zlib_raw(data, 1))
    return out


def fasta(rng, nbytes, dup=0.3):
    """random A/C/G/T records with 70-column lines, some copies of recent records"""
    recs, parts, size, i = [], [], 0, 0
    while size < nbytes:
        if recs and rng.random() < dup:
            body = rng.choice(recs[-50:])
        else:
            body = bytes(rng.choice(b"ACGT") for _ in range(rng.randint(200, 1200)))
            recs.append(body)
        r = b">seq_%d sample=S%d len=%d\n" % (i, i % 7, len(body)) + b"\n".join(body[k:k + 70] for k in range(0, len(body), 70)) + b"\n"
        parts.append(r)
        size += len(r)
        i += 1
    return b"".join(parts)[:nbytes]


def np_fasta(seed, nbytes):
    """a large FASTA-like text quickly: random bases, a newline every 71 bytes, a repeated block every 256 KiB"""
    g = np.random.default_rng(seed)
    a = np.frombuffer(b"ACGT", dtype=np.uint8)[g.integers(0, 4, nbytes)]
    a[70::71] = ord("\n")
    for k in range(1 << 18, nbytes - 30000, 1 << 18):
        a[k:k + 20000] = a[k - 25000:k - 5000]
    return a.tobytes()


@pytest.mark.parametrize("n", [1, 2, 3, 257, 258, 259, SEG - 1, SEG, SEG + 1, 3 * SEG + 17])
def test_sizes(ctx, n):
    rng = random.Random(n)
    check(ctx, fasta(rng, n))
    check(ctx, bytes(rng.getrandbits(8) for _ in range(min(n, 5000))) * (n // 5000 + 1))


def test_largest_call_and_one_more(ctx):
    from circkit_b200.core import CircKitError
    data = np_fasta(1, MAX)
    check(ctx, data)
    with pytest.raises(CircKitError) as e:
        ctx.deflate_submit(0, np.zeros(MAX + 1, dtype=np.uint8))
    assert e.value.code == -2
    check(ctx, data[:1000])                               # the slot is still usable


def test_argument_and_state_errors(ctx):
    from circkit_b200.core import CircKitError
    for args in [(b"",), (b"A", b"x" * 32769)]:
        with pytest.raises(CircKitError) as e:
            ctx.deflate_submit(1, *args)
        assert e.value.code == -2
    with pytest.raises(CircKitError) as e:
        ctx.deflate_wait(1)
    assert e.value.code == -3
    ctx.deflate_submit(1, b"ACGT" * 100)
    with pytest.raises(CircKitError) as e:
        ctx.deflate_submit(1, b"ACGT")
    assert e.value.code == -3
    out, crc = ctx.deflate_wait(1)
    assert zlib.decompressobj(-15).decompress(out) == b"ACGT" * 100


def test_contents(ctx):
    z = check(ctx, bytes(1 << 20))                        # length 258 at distance 1
    assert len(z) < 4000
    rnd = os.urandom(1 << 20)                             # stored blocks
    out = check(ctx, rnd)
    assert len(out) <= len(_zlib_raw(rnd, 1)) * 1.001
    check(ctx, bytes(range(256)) * 4096)
    rng = random.Random(5)
    for p in range(1, 301):
        unit = bytes(rng.getrandbits(8) for _ in range(p))
        out = check(ctx, (unit * (6000 // p + 2))[:6000])
        assert len(out) < 6000 // 2 + p + 64


def test_match_distances_at_the_window_edge(ctx):
    rng = random.Random(9)
    rec = b">dup\n" + bytes(rng.choice(b"ACGT") for _ in range(600)) + b"\n"
    for d in (32767, 32768, 32769):
        filler = fasta(rng, d - len(rec), dup=0)
        data = rec + filler + rec + fasta(rng, 5000, dup=0)
        assert data.index(rec, 1) == d
        check(ctx, data)
    # copies that straddle segment boundaries and whose source lies in the previous segment
    base = fasta(rng, 4 * SEG, dup=0)
    parts = bytearray(base)
    for k in (1, 2, 3):
        parts[k * SEG - 300:k * SEG + 300] = base[k * SEG - 10000:k * SEG - 9400]
    check(ctx, bytes(parts))


def test_matches_into_the_dictionary(ctx):
    rng = random.Random(3)
    dct = fasta(rng, 32768, dup=0)
    data = dct[1000:9000] + fasta(rng, 3000, dup=0) + dct[-5000:]
    with_dict = check(ctx, data, dct, crc=zlib.crc32(dct))
    alone = check(ctx, data)
    assert len(with_dict) < len(alone) // 2
    check(ctx, data, dct[-100:], crc=12345)


def test_both_slots_and_repeat_are_deterministic(ctx):
    rng = random.Random(11)
    a, b = fasta(rng, 700000), np_fasta(2, 3 << 20)
    ctx.deflate_submit(0, a)
    ctx.deflate_submit(1, b, a[-32768:], 77)
    ob, cb = ctx.deflate_wait(1)
    oa, ca = ctx.deflate_wait(0)
    assert (oa, ca) == ctx.deflate(a)
    assert (ob, cb) == ctx.deflate(b, a[-32768:], 77)
    assert zlib.decompressobj(-15).decompress(oa + ob) == a + b
    assert ca == zlib.crc32(a) and cb == zlib.crc32(b, 77)


def test_writer_stream_of_uneven_writes(tmp_path):
    from circkit_b200 import cli
    rng = random.Random(2)
    text = fasta(rng, 3 << 20)
    cuts = sorted(rng.sample(range(1, len(text)), 40))
    pieces = [text[i:j] for i, j in zip([0] + cuts, cuts + [len(text)])]
    pieces[3:3] = [b"", text[:1], b""]
    path = str(tmp_path / "w.fa.gz")
    w = cli.Writer(path, gzip_encoder=cli.DeviceDeflate())
    for p in pieces:
        w.write(p)
    w.close()
    want = b"".join(pieces)
    x = open(path, "rb").read()
    assert x[:10] == cli.GZIP_HEADER
    assert gzip.decompress(x) == want and zlib.decompress(x, 31) == want
    if shutil.which("gzip"):
        subprocess.run(["gzip", "-t", path], check=True)


def _cli_gz(tmp_path, argv, src, tag):
    """run argv on src with -o plain and -o .gz (twice); -> (plain bytes, gz bytes)"""
    from circkit_b200 import cli
    plain, gz1, gz2 = (str(tmp_path / ("%s%s" % (tag, s))) for s in (".fa", "1.fa.gz", "2.fa.gz"))
    extra = lambda o: ["--table", o + ".tsv"] if "--table" in argv else []     # noqa: E731
    args = [a for a in argv if a != "--table"]
    for o in (plain, gz1, gz2):
        assert cli.main(args[:1] + [src, "-o", o] + args[1:] + extra(o)) == 0
    g1, g2 = open(gz1, "rb").read(), open(gz2, "rb").read()
    assert g1 == g2
    p = open(plain, "rb").read()
    assert gzip.decompress(g1) == p and zlib.decompress(g1, 31) == p
    if "--table" in argv:
        assert open(gz1 + ".tsv", "rb").read() == open(plain + ".tsv", "rb").read()
    return p, g1


def test_cli_gz_output_equals_plain_output_and_the_goldens(tmp_path, monkeypatch, capsys):
    from circkit_b200 import cli
    from oracle import cli as ocli
    monkeypatch.setattr(cli, "MAX_BATCH_BYTES", 4096)      # many batches: many writes, many fragments
    monkeypatch.setattr(cli, "MAX_BATCH_RECORDS", 16)
    rep = os.path.join(FIX, "repeated", "in.fasta")
    p, _ = _cli_gz(tmp_path, ["canonicalize"], rep, "c")
    assert p == open(os.path.join(GOLD, "repeated.canonicalize.out"), "rb").read()
    p, _ = _cli_gz(tmp_path, ["uniq", "-c", "--table"], rep, "u")
    assert p == open(os.path.join(GOLD, "repeated.uniq_c.out"), "rb").read()
    rng = random.Random(21)
    src = str(tmp_path / "in.fa")
    data = fasta(rng, 300000)
    open(src, "wb").write(data)
    p, _ = _cli_gz(tmp_path, ["canonicalize"], src, "sc")
    assert p == ocli.cli_canonicalize(data)
    p, _ = _cli_gz(tmp_path, ["uniq", "-c", "--table"], src, "su")
    assert p == ocli.cli_uniq(data, canonicalize=True, table_ext="tsv")[0]
    mono = b"".join(b">m%d\n%s\n" % (i, (u * 3)[:len(u) * 2 + 7]) for i, u in
                    enumerate(bytes(rng.choice(b"ACGT") for _ in range(rng.randint(30, 200))) for _ in range(400)))
    msrc = str(tmp_path / "mono.fa")
    open(msrc, "wb").write(mono)
    p, _ = _cli_gz(tmp_path, ["monomerize"], msrc, "m")
    assert p == ocli.cli_monomerize(mono)[0]
    cap = capsys.readouterr()
    assert cap.out == "" and cap.err == ""


def test_large_inputs_beat_zlib_level_1(ctx):
    for data in (np_fasta(7, 8 << 20), fasta(random.Random(8), 2 << 20)):
        out = check(ctx, data)
        assert len(out) <= len(_zlib_raw(data, 1))
