"""CPU-side checks of the monomerize batch API's boundary: the layout of ck_mono_options as a C compiler sees it equals the
ctypes structure of the Python binding, and the Rust crate declares the same calls and the same fields in the same order."""
import ctypes
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ["seed_len", "flags", "overlap_dist", "overlap_min_identity", "min_length", "max_length", "min_overlap",
          "min_overlap_percent"]


@pytest.mark.skipif(shutil.which("gcc") is None, reason="needs gcc")
def test_c_layout_matches_the_ctypes_structure(tmp_path):
    from circkit_b200._native import CkMonoOptions
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "circkit_b200.h"\nint main(void) {\n'
                   '    printf("%zu\\n", sizeof(ck_mono_options));\n'
                   + "".join('    printf("%%zu\\n", offsetof(ck_mono_options, %s));\n' % f for f in FIELDS)
                   + '    printf("%u\\n", (unsigned)CK_MONO_KEEP_ALL);\n    return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert [f[0] for f in CkMonoOptions._fields_] == FIELDS
    assert got[0] == ctypes.sizeof(CkMonoOptions)
    assert got[1:-1] == [getattr(CkMonoOptions, f).offset for f in FIELDS]
    from circkit_b200 import _native
    assert got[-1] == _native.CK_MONO_KEEP_ALL


def test_rust_crate_declares_the_calls_and_the_fields():
    rs = open(os.path.join(ROOT, "circkit-cuda", "src", "lib.rs")).read()
    for fn in ("ck_mono_submit", "ck_mono_wait"):
        assert re.search(r"pub fn %s\(" % fn, rs), fn
    m = re.search(r"#\[repr\(C\)\][^{]*pub struct MonoOptions \{(.*?)\}", rs, re.S)
    assert m, "MonoOptions is not #[repr(C)]"
    names = re.findall(r"pub (\w+):", m.group(1))
    assert names == FIELDS
    types = re.findall(r"pub \w+: (\w+),", m.group(1))
    assert types == ["u32", "u32", "u64", "f64", "u64", "u64", "u64", "f64"]


def test_mono_options_are_checked_on_the_host():
    from circkit_b200 import cli
    for kw, msg in ((dict(seed_length=64), "at most 63"), (dict(seed_length=0), "at most 63"),
                    (dict(max_mismatch=1, min_identity=0.9), "both max_mismatch and min_identity"),
                    (dict(min_identity=1.5), "between 0.0 and 1.0"), (dict(min_overlap=-1), "negative")):
        with pytest.raises(cli.CliError, match=msg):
            cli.mono_options(**kw)
    o = cli.mono_options(sensitive=True, keep_all=True)
    assert (o.seed_len, o.flags, o.overlap_dist, o.overlap_min_identity, o.min_length, o.max_length, o.min_overlap) == \
        (10, 1 | 4, 0, -1.0, 0, 2**64 - 1, 0)
    assert o.min_overlap_percent != o.min_overlap_percent          # NaN = unset


def test_seed_64_fails_before_the_output_exists(tmp_path):
    from circkit_b200 import cli
    src = tmp_path / "in.fa"
    src.write_bytes(b">a\nACGT\n")
    dst = tmp_path / "out.fa"
    assert cli.main(["monomerize", str(src), "-o", str(dst), "--seed-length", "64"]) == 1
    assert not dst.exists()
    assert cli.main(["monomerize", str(tmp_path / "missing.fa"), "-o", str(dst)]) == 1
    assert not dst.exists()
