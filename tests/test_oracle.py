"""Pins the CPU oracle (oracle/) against the reference's own known answers and fixtures.

Mirrors lib/src/canonicalize.rs:65-232 (unit + proptest properties) and
tests/canon_uniq.rs / tests/compression.rs (fixtures, compared with the reference's own
order-insensitive id->seq comparator, tests/common.rs:33-88).
"""
import json
import os
import random

import pytest
from hypothesis import given, settings, strategies as st

import oracle
from oracle import cli

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
KATS = json.load(open(os.path.join(GOLDEN, "kats.json")))


# ---------------------------------------------------------------- unit KATs
@pytest.mark.parametrize("k", KATS["lmsr_index"], ids=lambda k: k["in"])
def test_lmsr_index_kat(k):
    assert oracle.lmsr_index(k["in"].encode()) == k["out"]


@pytest.mark.parametrize("k", KATS["lmsr"], ids=lambda k: k["in"])
def test_lmsr_kat(k):
    assert oracle.lmsr(k["in"].encode()) == k["out"].encode()


def test_lmsr_second_application_is_identical():      # lib/src/canonicalize.rs:102-106
    for s in KATS["lmsr_idempotent"]:
        t = oracle.lmsr(s.encode())
        assert oracle.lmsr(t) == t


@pytest.mark.parametrize("k", KATS["canonicalize"], ids=lambda k: k["in"])
def test_canonicalize_kat(k):
    assert oracle.canonicalize(k["in"].encode()) == k["out"].encode()


def test_real_monomer_rotations_agree():               # lib/src/canonicalize.rs:122-132
    for a, b in KATS["same_circle"]:
        assert oracle.lmsr(a.encode()) == oracle.lmsr(b.encode())
        assert oracle.canonicalize(a.encode()) == oracle.canonicalize(b.encode())
        assert oracle.canonicalize(a.encode()) == b"AAACGCTGCTAAATCAATTTCCTCCATCACCTAGTTTATGTAG"


def test_empty_and_single():
    assert oracle.lmsr_index(b"") == 0
    assert oracle.lmsr(b"") == b""
    assert oracle.canonicalize(b"") == b""
    assert oracle.canonicalize(b"T") == b"A"
    assert oracle.canonicalize(b"A") == b"A"
    assert oracle.canonicalize(b"N") == b"N"


# ---------------------------------------------------------------- proptest properties (:216-231)
printable = st.text(alphabet=[chr(c) for c in range(0x20, 0x7F)], min_size=1, max_size=100)


@settings(max_examples=400, deadline=None)
@given(printable)
def test_lmsr_index_implementations_are_identical(s):
    b = s.encode()
    assert oracle.lmsr_index_2(b) == oracle.lmsr_index_simple(b)
    assert oracle.lmsr_index_2(b) == oracle.lmsr_index(b)


@settings(max_examples=300, deadline=None)
@given(printable)
def test_lmsr_is_idempotent(s):
    b = s.encode()
    assert oracle.lmsr(oracle.lmsr(b)) == oracle.lmsr(b)


@settings(max_examples=300, deadline=None)
@given(st.text(alphabet="ATGC", min_size=1, max_size=100))
def test_canonicalize_is_idempotent(s):
    b = s.encode()
    assert oracle.canonicalize(oracle.canonicalize(b)) == oracle.canonicalize(b)


@settings(max_examples=300, deadline=None)
@given(st.text(alphabet="AC", min_size=1, max_size=40), st.integers(1, 6))
def test_periodic_strings_smallest_index(s, k):
    # tie rule: among equal minimal rotations the SMALLEST index wins (SURVEY §8 a1)
    b = (s * k).encode()
    assert oracle.lmsr_index(b) == oracle.lmsr_index_simple(b)


def test_faithful_cost_twin_same_answer():
    rng = random.Random(5)
    for _ in range(200):
        n = rng.randint(1, 120)
        b = bytes(rng.choice(b"ACGT") for _ in range(n))
        assert oracle.lib().ck_o_lmsr_index_faithful_cost(b, n) == oracle.lmsr_index(b)


def test_canonical_start_strand_consistent():
    rng = random.Random(7)
    comp = oracle.complement_table()
    for _ in range(500):
        n = rng.randint(1, 90)
        alpha = rng.choice([b"ACGT", b"AC", b"ACGTN-", b"ACGTRYKMacgtn"])
        s = bytes(rng.choice(alpha) for _ in range(n))
        if rng.random() < 0.3:
            s = s[: max(1, n // 3)] * 3
            n = len(s)
        start, strand = oracle.canonical_start(s)
        c = oracle.canonicalize(s)
        if strand == 0:
            rebuilt = bytes(s[(start + j) % n] for j in range(n))
        else:
            rebuilt = bytes(comp[s[(start - j) % n]] for j in range(n))
        assert rebuilt == c


# ---------------------------------------------------------------- third-party restatements
def test_complement_table_pinned_pairs():
    t = oracle.complement_table()
    # pinned by the reference: A<->T (canonicalize_test::att), C<->G (fixture multiple_sequences)
    assert t[ord("A")] == ord("T") and t[ord("T")] == ord("A")
    assert t[ord("C")] == ord("G") and t[ord("G")] == ord("C")
    # bio 1.3.1 table (unpinned by the reference's tests)
    for a, b in zip("AGCTYRWSKMDVHBN", "TCGARYWSMKHBDVN"):
        assert t[ord(a)] == ord(b)
        assert t[ord(a) + 32] == ord(b) + 32
    for c in b"U-u.*xz0 \n":
        assert t[c] == c


def test_normalize_rules():
    assert oracle.normalize(b"ACGTN-") == b"ACGTN-"
    assert oracle.normalize(b"acgtun") == b"ACGTTN"          # lowercase n -> "everything else" -> N
    assert oracle.normalize(b"AU.~ \t\r\nRYKMSWBDHVryk*x") == b"AT--" + b"N" * 15
    assert oracle.normalize(b"TT\nATG") == b"TTATG"          # fixture multiple_sequences_split_lines
    assert oracle.normalize(b"") == b""


def test_xxh3_against_python_xxhash_vectors():
    v = json.load(open(os.path.join(GOLDEN, "xxh3_vectors.json")))
    for k, h in v["known"].items():
        assert "%016x" % oracle.xxh3_64(k.encode()) == h
    for e in v["vectors"]:
        L = e["len"]
        if e["kind"] == "dna":
            data = bytes(b"ACGT"[(i * 7 + (i >> 3) * 3 + L) & 3] for i in range(L))
        else:
            data = bytes((i * 131 + 17 + L) & 0xFF for i in range(L))
        assert "%016x" % oracle.xxh3_64(data) == e["xxh3_64"], (L, e["kind"])


def test_xxh3_against_live_xxhash_if_present():
    # random bytes against python-xxhash's digests of them, stored by make_golden.py; and against python-xxhash itself
    # where it is installed
    try:
        import xxhash
    except ImportError:
        xxhash = None
    v = json.load(open(os.path.join(GOLDEN, "xxh3_vectors.json")))
    assert [e["len"] for e in v["random_vectors"]] == list(range(0, 300)) + [1023, 1024, 1025, 2048, 4097, 70000]
    rng = random.Random(11)
    for e in v["random_vectors"]:
        L = e["len"]
        data = bytes(rng.getrandbits(8) for _ in range(L))
        assert "%016x" % oracle.xxh3_64(data) == e["xxh3_64"], L
        if xxhash is not None:
            assert oracle.xxh3_64(data) == xxhash.xxh3_64_intdigest(data), L


# ---------------------------------------------------------------- CLI fixtures
def _id_seq_map(fasta: bytes):
    # the reference's comparator, tests/common.rs:33-88: id -> sequence with line breaks removed
    return {r.id: r.seq.replace(b"\n", b"").replace(b"\r", b"") for r in cli.parse_fasta(fasta)}


def _fx(d, name):
    return open(os.path.join(GOLDEN, "fixtures", d, name), "rb").read()


@pytest.mark.parametrize("d", KATS["cli_fixtures"]["canonicalize"])
@pytest.mark.parametrize("threads", [1, 2, 4])
def test_cli_canonicalize_fixture(d, threads):
    out = cli.cli_canonicalize(_fx(d, "in.fasta"), threads=threads)
    assert _id_seq_map(out) == _id_seq_map(_fx(d, "out.fasta"))


@pytest.mark.parametrize("d", KATS["cli_fixtures"]["uniq"])
@pytest.mark.parametrize("threads", [1, 2, 4])
def test_cli_uniq_fixture(d, threads):
    out, _ = cli.cli_uniq(_fx(d, "in.fasta"), canonicalize=True, threads=threads)   # tests/canon_uniq.rs:69-71
    assert _id_seq_map(out) == _id_seq_map(_fx(d, "out.fasta"))


def test_cli_simple_to_stdout():                          # tests/canon_uniq.rs:19-31
    assert b">seq1\nAATGC" in cli.cli_canonicalize(b">seq1\nATGCA")


def test_cli_compressed_inputs_decode_to_the_plain_fixture():
    import bz2, gzip, lzma
    plain = _fx("compressed_input", "in.fasta")
    assert gzip.decompress(_fx("compressed_input", "in.fasta.gz")) == plain
    assert bz2.decompress(_fx("compressed_input", "in.fasta.bz2")) == plain
    assert lzma.decompress(_fx("compressed_input", "in.fasta.xz")) == plain


def test_cli_outputs_match_committed_oracle_goldens():
    # guards the oracle against silent drift: committed byte-exact outputs
    od = os.path.join(GOLDEN, "oracle_cli")
    for f in sorted(os.listdir(od)):
        d, kind = f.split(".", 1)
        data = _fx(d, "in.fasta")
        want = open(os.path.join(od, f), "rb").read()
        if kind == "canonicalize.out":
            got = cli.cli_canonicalize(data)
        elif kind == "uniq.out":
            got = cli.cli_uniq(data, canonicalize=False)[0]
        elif kind == "uniq_c.out":
            got = cli.cli_uniq(data, canonicalize=True)[0]
        else:
            got = cli.cli_uniq(data, canonicalize=True, table_ext="csv")[1]
        assert got == want, f


def test_uniq_raw_echo_keeps_line_breaks_and_table():
    data = b">a x\nTT\nATG\n>b\nCATAA\n>c\nGGG\n"
    out, table = cli.cli_uniq(data, canonicalize=False, table_ext="tsv")
    assert out == b">a x\nTT\nATG\n>c\nGGG\n"           # raw record.seq() echo, src/uniq.rs:57-59
    assert table == b"id\tduplicate_id\na\tb\n"
    out, table = cli.cli_uniq(b">a\nACGT\n>b\nGGGA\n", table_ext="csv")
    assert table == b""                                    # no duplicates -> empty file


def test_fasta_reader_edges():
    assert cli.parse_fasta(b"") == []
    assert cli.parse_fasta(b"\n\n") == []
    r = cli.parse_fasta(b"\n>h1 d\r\nAC\r\nGT\r\n>h2\n\n>h3")
    assert [(x.head, x.seq) for x in r] == [(b"h1 d", b"AC\r\nGT"), (b"h2", b""), (b"h3", b"")]
    with pytest.raises(cli.FastaError):
        cli.parse_fasta(b"ACGT\n>x\nA")
