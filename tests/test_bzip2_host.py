"""CPU-side checks of the device bzip2 encoder's interface (ck_bzip2_submit / ck_bzip2_wait) and of the CLI's bzip2
framing around it: the constants and signatures agree between the header, the Python binding and the Rust crate, and
cli.Writer, driven by a libbz2 stand-in that honours the call contract, writes the bytes of bz2.compress(all, 9) whatever
the sizes of the writes."""
import bz2
import os
import random
import re
import shutil
import subprocess

import pytest

from circkit_b200 import cli

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CONSTANTS = ["CK_BZIP2_MAX_BYTES"]
BLOCK_MAX = 899981                                       # libbzip2's nblockMAX at level 9


@pytest.mark.skipif(shutil.which("gcc") is None, reason="needs gcc")
def test_constants_and_signatures_agree_across_header_binding_and_crate(tmp_path):
    from circkit_b200 import _native
    src = tmp_path / "probe.c"
    src.write_text('#include <stdio.h>\n#include "circkit_b200.h"\nint main(void) {\n'
                   '    int (*submit)(ck_ctx *, int, const uint8_t *, uint64_t, int, uint32_t, uint32_t, uint32_t) = 0;\n'
                   '    int (*wait)(ck_ctx *, int, uint8_t *, uint64_t *, uint64_t *, uint32_t *, uint32_t *, uint32_t *) = 0;\n'
                   '    int (*stats)(ck_ctx *, int, float *, uint32_t *) = 0;\n'
                   '    uint64_t (*bound)(uint64_t) = 0;\n'
                   '    (void)sizeof(submit = ck_bzip2_submit); (void)sizeof(wait = ck_bzip2_wait);\n'
                   '    (void)sizeof(stats = ck_bzip2_stats); (void)sizeof(bound = ck_bzip2_bound);\n'
                   + "".join('    printf("%%llu\\n", (unsigned long long)%s);\n' % c for c in CONSTANTS)
                   + '    return 0;\n}\n')
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-Wno-unused-but-set-variable", "-I", os.path.join(ROOT, "include"),
                    "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [64 << 20]
    assert got == [getattr(_native, c) for c in CONSTANTS]
    rs = open(os.path.join(ROOT, "circkit-cuda", "src", "lib.rs")).read()
    for c, v in zip(CONSTANTS, got):
        m = re.search(r"pub const %s: u(?:32|64) = ([0-9_x<() ]+);" % c, rs)
        assert m and eval(m.group(1).replace("_", "")) == v, c
    for fn in ("ck_bzip2_bound", "ck_bzip2_submit", "ck_bzip2_wait", "ck_bzip2_stats"):
        assert re.search(r"pub fn %s\(" % fn, rs), fn
        assert fn in _native.SIGNATURES
    assert len(_native.SIGNATURES["ck_bzip2_submit"][1]) == 8 and len(_native.SIGNATURES["ck_bzip2_wait"][1]) == 8


def rle1_tokens(data: bytes):
    """(raw start, raw length, RLE1 bytes) of bzip2's first stage: runs of one byte value split at 255"""
    out, i, n = [], 0, len(data)
    while i < n:
        e = i + 1
        while e < n and e - i < 255 and data[e] == data[i]:
            e += 1
        out.append((i, e - i, e - i if e - i < 4 else 5))
        i = e
    return out


def _bits(b: bytes) -> str:
    return bin(int.from_bytes(b, "big"))[2:].zfill(8 * len(b)) if b else ""


def block_bits(raw: bytes) -> "tuple[str, int]":
    """the one block of bz2.compress(raw, 9) as a bit string, and its CRC"""
    s = _bits(bz2.compress(raw, 9))
    crc = int(s[80:112], 2)
    for pad in range(8):
        e = len(s) - pad - 80
        if s[e:e + 48] == format(cli.BZIP2_EOS, "048b") and int(s[e + 48:e + 80], 2) == crc and "1" not in s[len(s) - pad:]:
            return s[32:e], crc
    raise AssertionError("no single block")


class Bz2StandIn:
    """What DeviceBzip2 promises, from libbz2: blocks cut by the RLE1 rule, each compressed alone (its raw range gives the
    same single block), packed after the pending bits; records every call"""

    def __init__(self, max_bytes):
        self.max_bytes, self.calls, self.closed = max_bytes, [], False

    def bzip2(self, data, final, bits, nbits, crc):
        data = bytes(data)
        self.calls.append((len(data), final))
        toks = rle1_tokens(data)
        if not final:
            toks = toks[:-1]                              # the last token may still grow
        s = format(bits, "0%db" % nbits) if nbits else ""
        consumed, acc, start = 0, 0, 0
        for k, (i, L, e) in enumerate(toks):
            acc += e
            if acc >= BLOCK_MAX or (final and k == len(toks) - 1):
                blk, bcrc = block_bits(data[start:i + L])
                s += blk
                crc = ((crc << 1 | crc >> 31) & 0xFFFFFFFF) ^ bcrc
                start = consumed = i + L
                acc = 0
        whole = len(s) // 8
        out = int(s[:8 * whole], 2).to_bytes(whole, "big") if whole else b""
        rest = s[8 * whole:]
        return out, consumed, int(rest, 2) if rest else 0, len(rest), crc

    def close(self):
        self.closed = True


class NoDevice:
    max_bytes = 1 << 20

    def bzip2(self, data, final, bits, nbits, crc):
        raise AssertionError("the encoder must not be called for an empty output")

    def close(self):
        pass


@pytest.mark.parametrize("max_bytes", [1 << 21, 3 << 20])
def test_writer_writes_libbz2_bytes(tmp_path, max_bytes):
    rng = random.Random(max_bytes)
    sizes = [0, 1, 7, 65536, 2000000, 0, 1, 7, 3100000, 1000]
    parts = []
    for n in sizes:                                       # FASTA-like text with runs, so the RLE1 cuts matter
        body = bytes(rng.choice(b"ACGT") for _ in range(min(n, 3000))) + b"A" * rng.randint(0, 600)
        parts.append(((b">r\n" + body + b"\n") * (n // (len(body) + 4) + 1))[:n])
    path = str(tmp_path / "o.fa.bz2")
    enc = Bz2StandIn(max_bytes)
    w = cli.Writer(path, bzip2_encoder=enc)
    for p in parts:
        w.write(p)
    w.close()
    want = b"".join(parts)
    assert open(path, "rb").read() == bz2.compress(want, 9)
    assert enc.closed
    assert all(0 < n <= max_bytes for n, _ in enc.calls) and [f for _, f in enc.calls].count(True) == 1
    assert len(enc.calls) >= 2


def test_stand_in_cuts_where_libbz2_does():
    rng = random.Random(3)
    x = bytes(rng.choice(b"ACGT\n") for _ in range(1900000)) + b"G" * 700 + bytes(rng.choice(b"AC") for _ in range(5000))
    enc = Bz2StandIn(1 << 30)
    out, consumed, bits, nbits, crc = enc.bzip2(x, True, 0, 0, 0)
    tail = (bits << 80 | cli.BZIP2_EOS << 32 | crc) << (-(nbits + 80) % 8)
    assert cli.BZIP2_HEADER + out + tail.to_bytes((nbits + 87) // 8, "big") == bz2.compress(x, 9)
    assert consumed == len(x)


def test_empty_output_is_the_14_byte_bz2(tmp_path):
    path = str(tmp_path / "e.bz2")
    w = cli.Writer(path, bzip2_encoder=NoDevice())
    w.write(b"")
    w.close()
    x = open(path, "rb").read()
    assert x == bz2.compress(b"", 9) and len(x) == 14


def test_cli_empty_input_to_bz2_needs_no_gpu(tmp_path, capsys):
    src = tmp_path / "empty.fa"
    src.write_bytes(b"")
    out = tmp_path / "x.bz2"
    assert cli.main(["canonicalize", str(src), "-o", str(out)]) == 0
    assert out.read_bytes() == bz2.compress(b"", 9)
    cap = capsys.readouterr()
    assert cap.out == "" and cap.err == ""


def test_writer_without_encoder_keeps_bz2file(tmp_path):
    path = str(tmp_path / "p.bz2")
    w = cli.Writer(path)
    assert isinstance(w.f, bz2.BZ2File)
    w.write(b">a\nACGT\n")
    w.close()
    assert bz2.decompress(open(path, "rb").read()) == b">a\nACGT\n"
