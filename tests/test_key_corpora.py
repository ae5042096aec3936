"""The planted-key corpora of tests/lane4_key_corpus.py (4-bit lane kernel) and tests/seg_key_corpus.py (segment kernel),
checked on the CPU before the GPU tests trust them: every family has the key occurrences, strands and kernel coordinates it
claims (brute force over all 2 n rotations), the sweeps cover every boundary they are meant to, the oracle picks the planted
rotation, and the CLI spelling of a record normalises back to it."""
from collections import defaultdict

import numpy as np
import pytest

import lane4_key_corpus as Q
import oracle
import seg_key_corpus as S


@pytest.fixture(scope="module")
def lane4():
    return Q.corpus()


@pytest.fixture(scope="module")
def mixed():
    return Q.mixed_batch()


@pytest.fixture(scope="module")
def seg():
    return S.corpus()


# ---------------------------------------------------------------- 4-bit lane corpus
def test_lane4_alphabet_and_complement(lane4):
    """{-, A, C, G, N, T} only; '-' and N complement to themselves in bio's table, as the corpus' reverse complement assumes"""
    comp = oracle.complement_table()
    assert [comp[c] for c in b"-ACGNT"] == list(b"-TGCNA")
    assert sorted(set(len(r.seq) for r in lane4)) == sorted(set(Q.SWEEP_LENGTHS) | set(Q.EDGE_LENGTHS))
    for r in lane4[::37]:
        assert Q.revcomp(r.seq) == oracle.revcomp(r.seq)
    assert all(set(r.seq) <= set(Q.ALPHA) for r in lane4)


def _lane4_key(r):
    return Q.key_value(b"--------" if r.k == 0 else b"---NN---") if r.family == 4 else Q.key_value(Q.KEY)


def test_lane4_family_claims(lane4, mixed):
    """declared occurrences == the brute-force set of rotations that begin with the minimal 8-mer, the number each family
    promises, the near miss where its `k` says, and the guard rule: the base in front of a planted key is not T on its strand
    (except "T-------A", where that T makes the second key)"""
    for r in lane4 + mixed:
        if not r.occ:
            assert r.family in (6, 8)
            continue
        n = len(r.seq)
        key, occ = Q.key_occurrences(r.seq)
        assert key == _lane4_key(r) and tuple(occ) == r.occ, (r.family, r.k, n, r.occ, occ[:6])
        nocc = len(occ)
        assert nocc == (1 if r.family in (1, 2, 7, 8) else 2 if r.family in (3, 4) else r.k), (r.family, r.k, nocc)
        if not (r.family == 3 and r.k == 4) and r.family != 4:
            for sd, st in occ:
                x = r.seq if sd == 0 else Q.revcomp(r.seq)
                assert x[(st - 1) % n] != ord("T"), (r.family, r.k, n, sd, st)
        (s1, a), *rest = occ
        if r.family == 2:
            near = Q.word_occurrences(r.seq, Q.NEAR)
            assert len(near) == 1 and Q.key_value(Q.NEAR) > key
            s2, b = near[0]
            assert (r.k == 0) == (s1 == s2 and a >> 6 == b >> 6) and (r.k == 1) == (s1 == s2 and a >> 6 != b >> 6)
            assert (r.k == 2) == (s1 != s2)
        elif r.family == 3:
            s2, b = rest[0]
            J1 = n >> 6
            want = {0: s1 != s2 and a >> 3 == b >> 3, 1: s1 == s2 and a >> 6 == b >> 6 and a >> 3 != b >> 3,
                    2: s1 == s2 and a >> 6 != b >> 6, 3: s1 != s2 and a >> 6 != b >> 6, 4: s1 != s2,
                    5: s1 == s2 and {a >> 6, b >> 6} == {J1, J1 - 1}, 6: s1 == s2 and max(a, b) > n - 8 and min(a, b) < 64}
            assert want[r.k], (r.k, n, occ)
        elif r.family == 4:
            assert s1 != rest[0][0]


def test_lane4_sweeps_cover_the_boundaries(lane4):
    """per sweep length and strand: every start residue mod 64, both edges of every oct and unit of one oct, the wrapping
    starts n - 8 .. n - 1, the last rotation of the partial oct and rotation 0; per length every near-miss and tie placement"""
    starts, fams = defaultdict(set), defaultdict(set)
    for r in lane4:
        n = len(r.seq)
        if r.family == 1:
            sd, st = r.occ[0]
            starts[(n, sd)].add(st)
        elif r.family in (2, 3, 4):
            fams[n].add((r.family, r.k))
    for n in Q.SWEEP_LENGTHS:
        J1 = n >> 6
        for sd in (0, 1):
            got = starts[(n, sd)]
            assert {p % 64 for p in got} == set(range(64)), (n, sd)
            assert {p % 8 for p in got if p >> 3 == (p + 1) >> 3} == set(range(7)), (n, sd)
            assert set(range(n - 8, n)) | {0} <= got
            assert {64 * j - 1 for j in range(1, J1 + 1)} | {64 * j for j in range(1, J1 + 1) if 64 * j < n} <= got, (n, sd)
            units = defaultdict(set)
            for p in got:
                units[p >> 6].add(p & 63)
            assert any({8 * u + e for u in range(8) for e in (0, 7)} <= v for v in units.values()), n
        ties = {k for f, k in fams[n] if f == 3}
        assert ties == set(range(7)) - ({5} if n & 63 < 10 else set()), (n, ties)
        assert {k for f, k in fams[n] if f == 2} == {0, 1, 2}
    assert {k for v in fams.values() for f, k in v if f == 4} == {0, 1}
    edge = defaultdict(set)
    for r in lane4:
        if r.family == 7:
            edge[len(r.seq)].add(r.occ[0][0])
    assert {n: v for n, v in edge.items()} == {n: {0, 1} for n in Q.EDGE_LENGTHS}


def test_lane4_oracle_picks_the_planted_rotation(lane4, mixed):
    """families with one minimal key: the canonical rotation is the key's (oracle.canonical_start: forward start, or
    n - 1 - start on the reverse strand)"""
    for r in lane4 + mixed:
        if r.family in (1, 2, 7, 8) and r.occ:
            n, (sd, st) = len(r.seq), r.occ[0]
            assert oracle.canonical_start(r.seq) == ((st, 0) if sd == 0 else (n - 1 - st, 1)), (r.family, n, r.occ)


def test_mixed_batch_pairs(mixed):
    """every pair (2 j, 2 j + 1) = the two halves of a k_pack4 warp holds one lane record and one the lane cannot take; the
    lane records sit at every byte offset residue mod 32, as the first and as the second of a pair"""
    off = np.concatenate([[0], np.cumsum([len(r.seq) for r in mixed])])
    res, halves, kinds = set(), set(), set()
    for j in range(0, len(mixed), 2):
        a, b = mixed[j], mixed[j + 1]
        assert bool(a.occ) != bool(b.occ)
        e, x, h = (a, b, 0) if a.occ else (b, a, 1)
        res.add(int(off[j + h]) % 32)
        halves.add(h)
        assert 129 <= len(e.seq) <= 2048 and set(e.seq) <= set(Q.ALPHA)
        if x.k == 0:
            assert len(x.seq) == len(e.seq) and set(x.seq) & set(Q.IUPAC)
        else:
            assert (len(x.seq) < 129) if x.k == 1 else (len(x.seq) > 2048)
        kinds.add(x.k)
    assert res == set(range(32)) and halves == {0, 1} and kinds == {0, 1, 2}


def test_cli_spelling_normalises_back(lane4):
    rng = np.random.default_rng(11)
    seen = set()
    for r in lane4[::5]:
        sp = Q.cli_spelling(r.seq, rng)
        assert oracle.normalize(sp) == r.seq
        seen |= set(sp)
    assert set(b".~-U\r \t") | set(b"acgtu") | set(Q.IUPAC) <= seen


# ---------------------------------------------------------------- segment corpus
def test_seg_geometry_matches_the_kernel_arithmetic():
    """scan_step / scan_lane / start_in_step restate ck_seg2.cuh: every rotation of either strand lies in exactly one step,
    the one locate's arithmetic numbers it by; lane ownership, and the lane counts of the examples in the kernel's terms"""
    for n in (8193, 8224, 8225, 8255, 9000, 16384):
        S1, per, lim, _ = S.geometry(n)
        for sd in (0, 1):
            seen = defaultdict(set)
            for t in range(S1 + 1):
                for s in range(32):
                    fwd_ok = s < lim if t == S1 else True
                    rev_ok = s >= 32 - lim if t == S1 else True
                    if (fwd_ok if sd == 0 else rev_ok):
                        seen[S.start_in_step(n, sd, t, s)].add(t)
            assert sorted(seen) == list(range(n)), (n, sd)
            assert all(len(v) == 1 for v in seen.values())
            assert all(S.scan_step(n, sd, st) == next(iter(t)) for st, t in seen.items()), (n, sd)
    assert (S.used_lanes(8193), S.used_lanes(16385), S.geometry(16385)[1]) == (22, 26, 5)
    for n, lanes, bl in ((8193, 9, 1), (32769, 17, 2), (425984, 32, 13)):
        C = (n + 15) >> 4
        assert S.geometry(n)[3] == bl and S.emit_lane(n, 16 * C - 1) == lanes - 1, n


def test_seg_family_claims(seg):
    """declared occurrences == every rotation of either strand whose 16-mer is A x 16 (brute force), the minimal key is A x 16,
    and the near misses and ties sit where their `k` says, in the kernel's steps and lanes"""
    for r in seg:
        n = len(r.seq)
        assert set(r.seq) <= set(b"ACGT")
        if not r.occ:
            assert r.family == 5
            continue
        key, occ = S.min_key_occurrences(r.seq)
        assert key == 0 and tuple(occ) == r.occ, (r.family, r.k, n, r.occ, occ[:6])
        S1 = S.geometry(n)[0]
        step = [S.scan_step(n, sd, st) for sd, st in occ]
        lane = [S.scan_lane(n, t) for t in step]
        if r.family == 1:
            assert len(occ) == 1
        elif r.family == 2:
            near = S.occurrences(r.seq, S.NEAR_VALUE)
            assert len(occ) == 1 and len(near) == 1, (n, near)
            t2 = S.scan_step(n, *near[0])
            want = {0: t2 == step[0], 1: t2 != step[0] and S.scan_lane(n, t2) == lane[0],
                    2: S.scan_lane(n, t2) != lane[0], 3: t2 == S1}
            assert want[r.k], (r.k, n, occ, near)
        elif r.family == 3:
            assert len(occ) == 2
            (s1, a), (s2, b) = occ
            want = {0: s1 == s2 and step[0] == step[1], 1: s1 != s2 and step[0] == step[1],
                    2: step[0] != step[1] and lane[0] == lane[1], 3: lane[0] != lane[1],
                    4: sorted(step) == [S1 - 1, S1], 5: s1 == s2 and (b - a) % n in (1, n - 1)}
            assert want[r.k], (r.k, n, occ, step, lane)
        else:
            assert len(occ) == r.k >= 3


def test_seg_sweeps_cover_the_boundaries(seg):
    """per length: the first and last rotation of every used scan lane (a sample at the long lengths), both strands; every
    residue mod 32 at three lengths; S1's last valid rotation and the first one past its mask; the wrapping starts; the record
    end at a 1024-base block edge -16, -1, 0, +1, +16; every near-miss and tie placement.  Across lengths: bl 1, 2 and 13,
    nfull % 16 of 0 and 15, both retry classes"""
    starts = defaultdict(set)
    fams = defaultdict(set)
    for r in seg:
        n = len(r.seq)
        if r.family == 1:
            sd, st = r.occ[0]
            starts[(n, sd)].add(st)
        elif r.family in (2, 3):
            fams[n].add((r.family, r.k))
    for n in S.LENGTHS:
        S1, per, lim, bl = S.geometry(n)
        for sd in (0, 1):
            got = starts[(n, sd)]
            edges = {(S.scan_step(n, sd, st), S.start_in_step(n, sd, S.scan_step(n, sd, st), 0) == st,
                      S.start_in_step(n, sd, S.scan_step(n, sd, st), 31) == st) for st in got}
            firsts = {S.scan_lane(n, t) for t, a, _ in edges if a and t == S.lane_steps(n, S.scan_lane(n, t))[0]}
            lasts = {S.scan_lane(n, t) for t, _, b in edges if b and t < S1 and t == S.lane_steps(n, S.scan_lane(n, t))[1]}
            need = set(range(S.used_lanes(n))) if n in S.FULL_SWEEP else {0, S.used_lanes(n) - 1}
            assert need <= firsts and need <= lasts, (n, sd, need - firsts, need - lasts)
            if n in S.RESIDUE_SWEEP:
                assert {st % 32 for st in got} == set(range(32)), (n, sd)
            wrap = set(range(n - 16, n)) if n <= 65537 else {n - 16, n - 15, n - 8, n - 2}
            assert wrap | {n - 1, 0} <= got, (n, sd)
            rel = {(n - st) % n for st in got}
            nblk = (((n + 15) >> 4) + 63) >> 6
            for d in (-16, -1, 0, 1, 16):
                ks = {k for k in range(1, nblk + 1) if (1024 * k - d) % n in rel}
                assert {1, nblk} <= ks and (n not in S.FULL_SWEEP or ks == set(range(1, nblk + 1))), (n, sd, d)
        rev = {S.window(n, 1, st) for st in starts[(n, 1)]}
        assert {0, 1} <= rev                                # S1's window n, and window 1 (step 0) just past its mask
        assert {k for f, k in fams[n] if f == 2} == {0, 1, 2, 3} and {k for f, k in fams[n] if f == 3} == set(range(6)), n
    assert {S.geometry(n)[3] for n in S.LENGTHS} >= {1, 2, 13}
    assert {((n - 1) >> 6) % 16 for n in S.LENGTHS} >= {0, 15}
    assert min(S.LENGTHS) == 8193 and max(S.LENGTHS) == 425984 and any(65536 < n for n in S.LENGTHS)


def test_seg_oracle_picks_the_planted_rotation(seg):
    for r in seg:
        if r.family in (1, 2) and (len(r.seq) <= 65537 or r.family == 2 or r.occ[0][1] % 7 == 0):
            n, (sd, st) = len(r.seq), r.occ[0]
            assert oracle.canonical_start(r.seq) == ((st, 0) if sd == 0 else (n - 1 - st, 1)), (r.family, n, r.occ)


def test_corpora_are_seeded_and_sized():
    a, b = Q.corpus(), Q.corpus()
    assert [r.seq for r in a] == [r.seq for r in b]
    total = sum(len(r.seq) for r in S.corpus())
    assert 60e6 < total <= 128 << 20
