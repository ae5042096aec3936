"""The tie corpus of tests/lane_tie_corpus.py, checked on the CPU before the GPU tests trust it: every family has the key
occurrences, strands, scan steps, first differing continuation base and wrap positions it claims (brute force over all 2 n
rotations), the sweeps cover what they are meant to, the numpy packer matches a per-base restatement of both packed2 arena
layouts, and the oracle picks the rotation the construction implies."""
from collections import defaultdict

import numpy as np
import pytest

import lane_tie_corpus as L
import oracle


@pytest.fixture(scope="module", params=["single", "doubled"])
def corpus(request):
    return request.param, (L.single_copy_corpus() if request.param == "single" else L.doubled_corpus())


def test_lengths(corpus):
    name, recs = corpus
    lens = sorted(set(len(r.seq) for r in recs))
    assert lens == (L.SINGLE_LENGTHS if name == "single" else L.DOUBLED_LENGTHS)
    assert all(set(r.seq) <= set(b"ACGT") for r in recs)
    assert 1500 < len(recs) < 8000


def test_family_properties(corpus):
    """declared occurrences == the brute-force set of rotations that begin with the minimal 8-mer (AAAAAAAA), and what each
    family promises about their number, strands and continuations"""
    _, recs = corpus
    for r in recs:
        if not r.occ:
            assert r.family in (0, 7)
            continue
        n = len(r.seq)
        key, occ = L.key_occurrences(r.seq)
        assert key == 0 and tuple(occ) == r.occ, (r.family, n, r.occ, occ[:8])
        strands = [sd for sd, _ in r.occ]
        if r.family == 1:
            assert len(occ) == 1
        elif r.family == 5:
            assert len(occ) >= 3
        else:
            assert len(occ) == 2
            assert L.first_difference(r.seq, *r.occ) == r.k, (r.family, n, r.occ)
            if r.family == 2:
                assert strands[0] == strands[1] and r.k < 16
            elif r.family == 3:
                assert strands == [0, 1] and r.k < 16
            elif r.family == 4:
                assert r.k == 16
            elif r.family == 6:
                assert r.k < 16 and any(n - 23 <= st <= n - 9 for _, st in r.occ)    # bases 8 .. 23 of one cross the end


def test_sweeps_cover_the_branches(corpus):
    """the lane kernel's cases, at lengths it takes (n >= 129): a single key in every window residue mod 32 and wrapping the
    end, on both strands; same-strand pairs in one scan step and in two, opposite-strand pairs and wrapping continuations, for
    every first differing base k = 0 .. 15"""
    _, recs = corpus
    cov = defaultdict(set)
    for r in recs:
        n = len(r.seq)
        if n < 129 or not r.occ:
            continue
        if r.family == 1:
            sd, st = r.occ[0]
            w = st if sd == 0 else (n - 8 - st) % n                 # forward window of the key
            cov[("window", sd)].add(w % 32)
            cov[("wrap", sd)].add(w - n if w >= n - 8 else None)
        elif r.family == 2:
            (s1, a), (s2, b) = r.occ
            cov[("pair", s1, L.kernel_step(n, s1, a) == L.kernel_step(n, s2, b))].add(r.k)
        elif r.family in (3, 6):
            cov[r.family].add(r.k)
    ks = set(range(16))
    for sd in (0, 1):
        assert cov[("window", sd)] == set(range(32))
        assert set(range(-8, 0)) <= cov[("wrap", sd)]
        assert cov[("pair", sd, True)] == ks and cov[("pair", sd, False)] == ks, sd
    assert cov[3] == ks and cov[6] == ks


def test_kernel_step_matches_the_scan_order():
    """kernel_step restates ck_stream2.cuh: step t sees forward starts 32 t .. 32 t + 31 and the reverse-strand keys of forward
    windows 32 t + 9 .. 32 t + 40, the last step ((n + 31) >> 5) - 1 also those of windows 0 .. 8"""
    for n in (129, 160, 200, 256, 300, 511, 512, 1025):
        last = ((n + 31) >> 5) - 1
        for p in range(n):
            assert L.kernel_step(n, 0, p) == p >> 5
        seen = defaultdict(list)
        for st in range(n):
            seen[L.kernel_step(n, 1, st)].append((n - 8 - st) % n)
        assert set(seen) == set(range(last + 1))
        for t, ws in seen.items():
            ext = sorted(w if w >= 9 else w + n for w in ws)
            assert ext == list(range(32 * t + 9, min(32 * t + 41, n + 9))), (n, t)


def test_pack2_matches_the_per_base_layout():
    """both layouts on every length 1 .. 600: unit j of record i holds bases 16 j .. 16 j + 15 (mod n), first base in bits
    31..30; records start at their granule; nothing else is written"""
    rng = np.random.default_rng(5)
    seqs = [rng.choice(np.frombuffer(b"ACGT", np.uint8), n).astype(np.uint8).tobytes() for n in range(1, 601)]
    code = {65: 0, 67: 1, 71: 2, 84: 3}
    for single in (True, False):
        off, arena = L.pack2(seqs, single)
        assert np.array_equal(off, np.concatenate([[0], np.cumsum([len(s) for s in seqs])]).astype(np.uint64))
        total, n_rec = int(off[-1]), len(seqs)
        assert arena.dtype == np.uint64 and len(arena) == (2 * ((total >> 6) + 2 * n_rec + 2) if single
                                                           else 4 * ((total >> 6) + 3 * n_rec + 3))
        units = arena.view(np.uint32)
        written = np.zeros(len(units), dtype=bool)
        for i, s in enumerate(seqs):
            n, o = len(s), int(off[i])
            u0 = 4 * ((o >> 6) + 2 * i) if single else 8 * ((o >> 6) + 3 * i)
            last = (n >> 4) + 4 if single else max((2 * n + 143) >> 4, (n >> 4) + 5)
            assert not written[u0: u0 + last + 1].any(), (single, i)         # records do not overlap
            written[u0: u0 + last + 1] = True
            for j in range(last + 1):
                u = int(units[u0 + j])
                for b in range(16):
                    assert (u >> (30 - 2 * b)) & 3 == code[s[(16 * j + b) % n]], (single, n, j, b)
        assert not units[~written].any()


def test_oracle_picks_the_constructed_rotation():
    """families 1, 2, 3 and 6 parse as intended: the canonical rotation is the key occurrence whose continuation is smaller
    (oracle.canonical_start: forward start, or n - 1 - start on the reverse strand)"""
    recs = [r for r in L.single_copy_corpus() if r.family in (1, 2, 3, 6)]
    for r in recs[::7]:
        n = len(r.seq)
        win = r.occ[0]
        if len(r.occ) == 2:
            a, b = (L.continuation(r.seq, *o)[r.k] for o in r.occ)
            win = r.occ[0] if a < b else r.occ[1]
        sd, st = win
        assert oracle.canonical_start(r.seq) == ((st, 0) if sd == 0 else (n - 1 - st, 1)), (r.family, n, r.occ, r.k)


def test_duplicates_collapse_onto_their_originals():
    rng = np.random.default_rng(3)
    seqs = [r.seq for r in L.single_copy_corpus()[::3]]
    allseqs = L.rotations_and_revcomps(seqs, rng)
    assert len(allseqs) > 1.3 * len(seqs)
    canon = {oracle.canonicalize(s) for s in seqs}
    assert all(oracle.canonicalize(s) in canon for s in allseqs[len(seqs):])
