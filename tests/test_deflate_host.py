"""CPU-side checks of the device DEFLATE encoder's interface (ck_deflate_submit / ck_deflate_wait) and of the CLI's gzip
framing around it: the constants and signatures agree between the header, the Python binding and the Rust crate, and
cli.Writer, driven by a zlib stand-in for the device encoder, writes one valid gzip member whatever the sizes of the
writes."""
import gzip
import os
import random
import re
import shutil
import subprocess
import zlib

import pytest

from circkit_b200 import cli

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CONSTANTS = ["CK_DEFLATE_MAX_BYTES", "CK_DEFLATE_DICT_BYTES"]


@pytest.mark.skipif(shutil.which("gcc") is None, reason="needs gcc")
def test_constants_and_signatures_agree_across_header_binding_and_crate(tmp_path):
    from circkit_b200 import _native
    src = tmp_path / "probe.c"
    src.write_text('#include <stdio.h>\n#include "circkit_b200.h"\nint main(void) {\n'
                   '    int (*submit)(ck_ctx *, int, const uint8_t *, uint64_t, const uint8_t *, uint32_t, uint32_t) = 0;\n'
                   '    int (*wait)(ck_ctx *, int, uint8_t *, uint64_t *, uint32_t *) = 0;\n'
                   '    uint64_t (*bound)(uint64_t) = 0;\n'
                   '    (void)sizeof(submit = ck_deflate_submit); (void)sizeof(wait = ck_deflate_wait); (void)sizeof(bound = ck_deflate_bound);\n'
                   + "".join('    printf("%%llu\\n", (unsigned long long)%s);\n' % c for c in CONSTANTS)
                   + '    return 0;\n}\n')
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-Wno-unused-but-set-variable", "-I", os.path.join(ROOT, "include"),
                    "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [64 << 20, 32768]
    assert got == [getattr(_native, c) for c in CONSTANTS]
    rs = open(os.path.join(ROOT, "circkit-cuda", "src", "lib.rs")).read()
    for c, v in zip(CONSTANTS, got):
        m = re.search(r"pub const %s: u(?:32|64) = ([0-9_x<() ]+);" % c, rs)
        assert m and eval(m.group(1).replace("_", "")) == v, c
    for fn in ("ck_deflate_bound", "ck_deflate_submit", "ck_deflate_wait"):
        assert re.search(r"pub fn %s\(" % fn, rs), fn
        assert fn in _native.SIGNATURES
    assert len(_native.SIGNATURES["ck_deflate_submit"][1]) == 7 and len(_native.SIGNATURES["ck_deflate_wait"][1]) == 5


class ZlibSyncEncoder:
    """What DeviceDeflate promises, from zlib: raw deflate of `data` with `dict` as the preset dictionary, ending in a sync
    flush; records every call"""

    def __init__(self, max_bytes):
        self.max_bytes, self.calls, self.closed = max_bytes, [], False

    def deflate(self, data, dict, crc):
        data = bytes(data)
        self.calls.append((data, dict, crc))
        c = zlib.compressobj(6, zlib.DEFLATED, -15, zdict=dict) if dict else zlib.compressobj(6, zlib.DEFLATED, -15)
        return c.compress(data) + c.flush(zlib.Z_SYNC_FLUSH), zlib.crc32(data, crc)

    def close(self):
        self.closed = True


class NoDevice:
    max_bytes = 1 << 20

    def deflate(self, data, dict, crc):
        raise AssertionError("the encoder must not be called for an empty output")

    def close(self):
        pass


def _one_member(x: bytes, want: bytes):
    assert x[:10] == cli.GZIP_HEADER
    assert zlib.decompress(x, 31) == want
    d = zlib.decompressobj(31)
    assert d.decompress(x) == want and d.eof and d.unused_data == b""
    assert gzip.decompress(x) == want


@pytest.mark.parametrize("max_bytes", [1 << 16, 1 << 20])
def test_writer_frames_one_gzip_member(tmp_path, max_bytes):
    rng = random.Random(max_bytes)
    sizes = [0, 1, 7, 65535, 65536, 200000, 0, 1, 7]
    parts = []
    for n in sizes:                                       # FASTA-like text with repeats, so the dictionaries matter
        body = bytes(rng.choice(b"ACGT") for _ in range(min(n, 3000)))
        parts.append(((b">r\n" + body + b"\n") * (n // (len(body) + 4) + 1))[:n])
    path = str(tmp_path / "o.fa.gz")
    enc = ZlibSyncEncoder(max_bytes)
    w = cli.Writer(path, gzip_encoder=enc)
    for p in parts:
        w.write(p)
    w.close()
    want = b"".join(parts)
    x = open(path, "rb").read()
    _one_member(x, want)
    assert enc.closed
    assert x[-8:] == zlib.crc32(want).to_bytes(4, "little") + (len(want) & 0xFFFFFFFF).to_bytes(4, "little")
    # every call gets at most max_bytes, the last 32 KiB before it as dictionary and the CRC so far
    done = b""
    for data, dct, crc in enc.calls:
        assert 0 < len(data) <= max_bytes
        assert dct == done[-32768:] and crc == zlib.crc32(done)
        done += data
    assert done == want


def test_empty_output_is_a_20_byte_gzip(tmp_path):
    path = str(tmp_path / "e.gz")
    w = cli.Writer(path, gzip_encoder=NoDevice())
    w.write(b"")
    w.close()
    x = open(path, "rb").read()
    assert len(x) == 20
    _one_member(x, b"")


def test_cli_empty_input_to_gz_needs_no_gpu(tmp_path, capsys):
    src = tmp_path / "empty.fa"
    src.write_bytes(b"")
    out = tmp_path / "x.gz"
    assert cli.main(["canonicalize", str(src), "-o", str(out)]) == 0
    x = out.read_bytes()
    assert len(x) == 20 and x[:10] == cli.GZIP_HEADER and gzip.decompress(x) == b""
    cap = capsys.readouterr()
    assert cap.out == "" and cap.err == ""


def test_writer_without_encoder_keeps_gzipfile(tmp_path):
    path = str(tmp_path / "p.gz")
    w = cli.Writer(path)
    assert isinstance(w.f, gzip.GzipFile)
    w.write(b">a\nACGT\n")
    w.close()
    assert gzip.decompress(open(path, "rb").read()) == b">a\nACGT\n"
