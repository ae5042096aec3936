"""CPU-side checks of the FASTA text batch API (ck_fasta_submit / ck_fasta_wait): its constants agree between the header,
the Python binding and the Rust crate, and the host's cut rule -- pieces of iter_text, batches of _text_batches -- never
splits a record, on random texts and on the reference fixtures."""
import os
import random
import re
import shutil
import subprocess

import numpy as np
import pytest

from circkit_b200 import cli

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIX = os.path.join(ROOT, "tests", "golden", "fixtures")
CONSTANTS = ["CK_CMD_CANONICALIZE", "CK_CMD_UNIQ", "CK_CMD_MONOMERIZE", "CK_F_CANONICAL_BODY"]


@pytest.mark.skipif(shutil.which("gcc") is None, reason="needs gcc")
def test_constants_agree_across_header_binding_and_crate(tmp_path):
    from circkit_b200 import _native
    src = tmp_path / "probe.c"
    # the declarations must have these types (-Werror: an incompatible pointer assignment fails); sizeof keeps the
    # assignments unevaluated, so nothing needs linking
    src.write_text('#include <stdio.h>\n#include "circkit_b200.h"\nint main(void) {\n'
                   '    int (*submit)(ck_ctx *, int, const uint8_t *, uint64_t, uint32_t, uint32_t, uint64_t, const ck_mono_options *,\n'
                   '                  uint32_t *) = 0;\n'
                   '    int (*wait)(ck_ctx *, int, uint8_t *, uint64_t *, uint32_t *, uint32_t *, uint64_t *, uint64_t *, uint32_t *,\n'
                   '                uint32_t *) = 0;\n'
                   '    uint64_t (*bound)(uint64_t, uint32_t) = 0;\n'
                   '    (void)sizeof(submit = ck_fasta_submit); (void)sizeof(wait = ck_fasta_wait); (void)sizeof(bound = ck_fasta_out_bytes);\n'
                   + "".join('    printf("%%llu\\n", (unsigned long long)%s);\n' % c for c in CONSTANTS)
                   + '    return 0;\n}\n')
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-Wno-unused-but-set-variable", "-I", os.path.join(ROOT, "include"),
                    "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [getattr(_native, c) for c in CONSTANTS]
    flags = [_native.CK_F_NORMALIZE, _native.CK_F_NO_BYTES, _native.CK_F_ALIGNED_OUT, _native.CK_F_PACKED_IN,
             _native.CK_F_SURVIVORS, _native.CK_F_SINGLE_COPY]
    assert _native.CK_F_CANONICAL_BODY not in flags                 # a flag bit of its own
    rs = open(os.path.join(ROOT, "circkit-cuda", "src", "lib.rs")).read()
    for c, v in zip(CONSTANTS, got):
        m = re.search(r"pub const %s: u32 = (\d+);" % c, rs)
        assert m and int(m.group(1)) == v, c
    for fn in ("ck_fasta_out_bytes", "ck_fasta_submit", "ck_fasta_wait"):
        assert re.search(r"pub fn %s\(" % fn, rs), fn
        assert fn in _native.SIGNATURES
    assert len(_native.SIGNATURES["ck_fasta_submit"][1]) == 9 and len(_native.SIGNATURES["ck_fasta_wait"][1]) == 10


def _random_text(rng, n):
    """records with CRLF / LF, wrapped lines, header-only and empty records, '>' inside sequence and header lines, leading
    blank lines, with or without a final newline"""
    recs = []
    for i in range(n):
        eol = rng.choice([b"\n", b"\r\n"])
        head = b"r%d%s" % (i, rng.choice([b"", b" a>b", b" \xc3\xa9"]))
        body = bytes(rng.choice(b"ACGT>") for _ in range(rng.randint(0, 90)))
        width = rng.choice([0, 5, 30])
        lines = [body[k: k + width] for k in range(0, len(body), width)] if width and body else [body]
        kind = rng.randrange(5)
        if kind == 0:
            recs.append(b">" + head)                          # header only, no line break
        elif kind == 1:
            recs.append(b">" + head + eol)
        else:
            recs.append(b">" + head + eol + eol.join(lines) + eol)
    text = rng.choice([b"", b"\n", b"\r\n\n"]) + b"\n".join(r.rstrip(b"\n") if i % 7 == 0 else r for i, r in enumerate(recs))
    return text if rng.random() < 0.5 else text.rstrip(b"\n")


def _starts(text):
    """absolute start of every record of a text, by cli.Records"""
    r = cli.Records(text)
    return (r.head_lo - 1).tolist()


def test_iter_text_cuts_where_iter_records_cuts():
    rng = random.Random(5)
    for trial in range(40):
        text = _random_text(rng, rng.randint(1, 60))
        chunk = rng.choice([1, 3, 17, 64, 1000])
        chunks = [text[k: k + chunk] for k in range(0, len(text), chunk)]
        pieces = list(cli.iter_text(chunks))
        assert b"".join(pieces) == text
        recs = list(cli.iter_records(chunks))
        assert [bytes(r.data) for r in recs] == pieces
        # every piece but the first begins at a record start, and the records of the pieces are those of the whole text
        want = _starts(text)
        got, base = [], 0
        for p in pieces:
            got += [base + s for s in _starts(p)]
            base += len(p)
        assert got == want


@pytest.mark.parametrize("max_bytes,max_records", [(1, 1), (40, 3), (200, 2), (10 ** 6, 4), (10 ** 6, 10 ** 6)])
def test_text_batches_never_split_a_record(max_bytes, max_records):
    rng = random.Random(max_bytes * 31 + max_records)
    texts = [_random_text(rng, rng.randint(1, 80)) for _ in range(25)]
    texts += [open(os.path.join(FIX, d, "in.fasta"), "rb").read() for d in sorted(os.listdir(FIX))
              if os.path.isfile(os.path.join(FIX, d, "in.fasta"))]
    for text in texts:
        text = cli._piece_text(text)
        if not text:
            continue
        want = _starts(text)
        got, cuts = [], list(cli._text_batches(text, max_bytes, max_records, oversize=True))
        assert cuts[0][0] == 0 and cuts[-1][1] == len(text)
        for (lo, hi), nxt in zip(cuts, cuts[1:] + [(len(text), None)]):
            assert hi == nxt[0] and text[lo:lo + 1] == b">"
            s = _starts(text[lo:hi])
            assert len(s) <= max_records
            assert hi - lo <= max_bytes or len(s) == 1        # only a record longer than max_bytes stands alone
            assert text[lo:hi].count(b"\n>") + 1 == len(s)   # the record count the driver computes at C speed
            got += [lo + x for x in s]
        assert got == want


def test_a_record_longer_than_the_batch_is_an_error_without_oversize():
    text = b">a\nACGT\n>b\n" + b"A" * 100 + b"\n>c\nA\n"
    assert list(cli._text_batches(text, 1000, 10)) == [(0, len(text))]
    with pytest.raises(cli.FastaError, match="longer than the batch size"):
        list(cli._text_batches(text, 50, 10))
    assert list(cli._text_batches(text, 50, 10, oversize=True)) == [(0, 8), (8, 112), (112, len(text))]


def test_piece_text_applies_the_leading_blank_line_rule():
    assert cli._piece_text(b"\n\r\n>a\nAC\n") == b">a\nAC\n"
    assert cli._piece_text(b"\r") == b"" and cli._piece_text(b"") == b""
    for bad in (b"ACGT\n>a\n", b"\n \n>a\n", b"\r\r\n>a\n"):
        with pytest.raises(cli.FastaError, match="expected '>'"):
            cli._piece_text(bad)
        with pytest.raises(cli.FastaError, match="expected '>'"):
            cli.Records(bad)
    r = cli.Records(b"\n>a\nAC\n>b\n")
    assert cli._piece_text(r) == b">a\nAC\n>b\n"
    assert np.array_equal(cli.Records(cli._piece_text(r)).head_lo, r.head_lo - 1)
