"""2-bit records of 8 193 .. 425 984 bases built on purpose for the segment kernel (k_canon_seg, ck_seg2.cuh).  Helper of
tests/test_key_corpora.py and tests/test_gpu_segment_keys.py; it holds no tests.

The kernel's keys are 16-mers.  Every family plants KEY = A x 16 into lane_tie_corpus._bg's background (over {C, G, T}, its
T-runs at most 3, so neither strand has an A-run of its own); a reverse-strand key is a planted T x 16; a planted key has C in front
of it and G after it on its strand.  Occurrences are (strand, start) in the strand's own coordinates; a reverse-strand record of a family is the
reverse complement of a forward construction.

Where the kernel sees an occurrence (`scan_step`, `scan_lane`, restating ck_seg2.cuh): S1 = ceil(n / 32) - 1 is the partial
step, octs = (S1 + 4) >> 2, per = ceil(octs / 32); lane l scans the full steps [4 l per, 4 (l + 1) per) and lane 0 also S1.
A forward start p is in step p >> 5; a reverse-strand key whose forward window starts at f (f = n for window 0) is in step
(f - 1) >> 5.  The emit pass (`emit_lane`) cuts the canonical string into 1024-base blocks, bl = ceil(ceil(ceil(n / 16) /
64) / 32) of them per lane; the record end lies at offset (n - start) mod n of the canonical string.

Families (`Rec.family`):
  1  one key; its start at the first and last rotation of every used scan lane (a sample at the long lengths), every residue
     mod 32, the last valid rotation of S1 and the first one past its mask (forward: n - 1 and 0; reverse: windows n and 1),
     n - 16 .. n - 1 (wrapping), and the starts n - 1024 k + {-16, -1, 0, 1, 16} that put the record end next to a block
     edge; both strands;
  2  one key and the near miss A x 15 C: `k` 0 same step, 1 same lane, 2 another lane, 3 the near miss in S1;
  3  two keys: `k` 0 same step and strand, 1 same step, opposite strands, 2 same lane, different steps, 3 different lanes,
     4 one in S1 and one in the last full step, 5 an A-run of 17;
  4  three or more keys;
  5  structure: lane_tie_corpus.structured's shapes and random records (`occ` not declared).
"""
from __future__ import annotations

import numpy as np

from lane_tie_corpus import Rec, _bg, _finish, _put, pack2, revcomp, rotations_and_revcomps, structured  # noqa: F401

KEY = b"A" * 16
NEAR = b"A" * 15 + b"C"
LENGTHS = [8193, 8224, 8225, 8255, 12289, 16384, 16385, 32768, 32769, 33793, 65536, 65537, 131073, 262143, 425984]
FULL_SWEEP = (8193, 8224, 8225, 8255, 12289, 16384, 16385)    # every used scan lane; the longer lengths get a sample
RESIDUE_SWEEP = (8193, 16385, 65537)                          # every residue mod 32
TIE_FAMILIES = (3, 4)
_CODE = np.full(256, 255, dtype=np.uint8)
_CODE[list(b"ACGT")] = [0, 1, 2, 3]


# ---------------------------------------------------------------- the kernel's coordinates
def geometry(n: int):
    """-> (S1, per, lim, bl): partial step, octs per scan lane, valid rotations of S1, 1024-base blocks per emit lane"""
    S1 = ((n + 31) >> 5) - 1
    octs = (S1 + 4) >> 2
    C = (n + 15) >> 4
    return S1, (octs + 31) >> 5, n - 32 * S1, (((C + 63) >> 6) + 31) >> 5


def window(n: int, strand: int, start: int) -> int:
    """forward position of the first base of occurrence (strand, start)"""
    return start if strand == 0 else (n - 16 - start) % n


def scan_step(n: int, strand: int, start: int) -> int:
    if strand == 0:
        return start >> 5
    f = window(n, 1, start) or n
    return (f - 1) >> 5


def scan_lane(n: int, step: int) -> int:
    S1, per, _, _ = geometry(n)
    return 0 if step == S1 else step // (4 * per)


def used_lanes(n: int) -> int:
    S1, per, _, _ = geometry(n)
    return (S1 + 4 * per - 1) // (4 * per)


def emit_lane(n: int, offset: int) -> int:
    """the emit lane that writes canonical offset `offset`"""
    return (offset >> 10) // geometry(n)[3]


def lane_steps(n: int, lane: int) -> tuple[int, int]:
    """first and last full step of a scan lane"""
    S1, per, _, _ = geometry(n)
    return 4 * per * lane, min(4 * per * (lane + 1), S1) - 1


def start_in_step(n: int, strand: int, step: int, s: int) -> int:
    """the start of rotation s (0 .. 31) of a step, as locate numbers it: forward 32 t + s, reverse n - 48 - 32 t + s"""
    return (32 * step + s) % n if strand == 0 else (n - 48 - 32 * step + s) % n


# ---------------------------------------------------------------- families
def footprint(n: int, strand: int, start: int, length: int = 16) -> set:
    f = window(n, strand, start)
    return {(f - 1 + i) % n for i in range(length + 2)}


def _plant(s: bytearray, strand: int, start: int, word: bytes):
    """word at (strand, start) as C + word + G on its strand: no A-run grows past 16, and the key is not followed by a C
    (A x 15 C, the near miss, would start one base later)"""
    n = len(s)
    f = window(n, strand, start)
    _put(s, f - 1, b"C" + word + b"G" if strand == 0 else revcomp(b"C" + word + b"G"))


def _planted(rng, n: int, plants, family: int, k=None, reverse: bool = False) -> Rec:
    used = set()
    for sd, st, w in plants:
        fp = footprint(n, sd, st)
        assert not fp & used, (n, plants)
        used |= fp
    s = _bg(rng, n)
    for sd, st, w in plants:
        _plant(s, sd, st, w)
    return _finish(s, [(sd, st) for sd, st, w in plants if w == KEY], family, k, reverse)


def one_key(rng, n: int, strand: int, start: int) -> Rec:
    """the key at (strand, start) of the record: built forward, reverse-complemented for strand 1"""
    return _planted(rng, n, [(0, start, KEY)], 1, None, strand == 1)


def sweep_starts(n: int, rng) -> list[int]:
    """family 1's starts (strand coordinates; the same for both strands)"""
    S1, per, lim, bl = geometry(n)
    lanes = range(used_lanes(n))
    if n not in FULL_SWEEP:
        lanes = sorted({0, 1, used_lanes(n) - 1} | set(int(x) for x in rng.integers(0, used_lanes(n), 3 if n <= 65537 else 1)))
    st = set()
    for ln in lanes:
        a, b = lane_steps(n, ln)
        st |= {start_in_step(n, 0, a, 0), start_in_step(n, 0, b, 31)}
    if n in RESIDUE_SWEEP:
        st |= {32 * int(rng.integers(S1)) + r for r in range(32)}
    st |= {n - 1, 0} | (set(range(n - 16, n)) if n <= 65537 else {n - 16, n - 15, n - 8, n - 2})
    nblk = (((n + 15) >> 4) + 63) >> 6
    ks = (range(1, nblk + 1) if n in FULL_SWEEP else {1, 2, nblk, int(rng.integers(3, nblk))} if n <= 65537
          else {1, nblk, int(rng.integers(2, nblk))})
    st |= {(n - 1024 * k + d) % n for k in ks for d in (-16, -1, 0, 1, 16)}
    return sorted(st)


def reverse_sweep(n: int, rng) -> list[int]:
    """reverse-strand starts of the lane edges, as the reverse strand's own scan sees them: first rotation (window 32 t + 32)
    of a lane's first step, last one (window 32 t + 1) of its last step; S1's window n and the first window past its mask, 1"""
    starts = []
    for ln in (range(used_lanes(n)) if n in FULL_SWEEP else (0, used_lanes(n) - 1)):
        a, b = lane_steps(n, ln)
        starts += [start_in_step(n, 1, a, 0), start_in_step(n, 1, b, 31)]
    return starts + [(n - 16) % n, (n - 17) % n]


def _in_steps(rng, n: int, draw, family: int, k, reverse: bool) -> Rec:
    """plants drawn as (strand, step, rotation s of the step, word) of the finished record, redrawn until their footprints are
    disjoint"""
    for _ in range(1000):
        plants = [(sd ^ reverse, start_in_step(n, sd, t, s), w) for sd, t, s, w in draw()]
        used = [footprint(n, sd, st) for sd, st, _ in plants]
        if sum(len(u) for u in used) == len(set().union(*used)):
            return _planted(rng, n, plants, family, k, reverse)
    raise AssertionError((n, family, k))


def _s1_rotation(rng, n: int, strand: int) -> int:
    """a rotation of the partial step S1 that its mask keeps: forward s < lim, reverse s >= 32 - lim"""
    lim = geometry(n)[2]
    return int(rng.integers(lim)) if strand == 0 else 32 - lim + int(rng.integers(lim))


def near_miss(rng, n: int, k: int, reverse: bool) -> Rec:
    S1, per, lim, _ = geometry(n)
    r32 = lambda: int(rng.integers(32))                    # noqa: E731
    sd = int(reverse)

    def draw():
        if k == 0:                                         # same step
            t = int(rng.integers(S1))
            a, b = (sd, t, r32()), (sd, t, r32())
        elif k == 1:                                       # same lane, different steps
            t = int(rng.integers(lane_steps(n, 0)[1]))
            a, b = (sd, t, r32()), (sd, t + 1, r32())
        elif k == 2:                                       # another lane
            ln = 1 + int(rng.integers(used_lanes(n) - 1))
            a, b = (sd, int(rng.integers(4 * per)), r32()), (sd, lane_steps(n, ln)[int(rng.integers(2))], r32())
        else:                                              # the near miss in S1 (its window wraps the end when lim < 16)
            a, b = (sd, int(rng.integers(S1 // 2)), r32()), (sd, S1, _s1_rotation(rng, n, sd))
            return [a + (KEY,), b + (NEAR,)]
        return [a + (KEY,), b + (NEAR,)] if k % 2 == 0 else [a + (NEAR,), b + (KEY,)]
    return _in_steps(rng, n, draw, 2, k, reverse)


def two_keys(rng, n: int, k: int, reverse: bool) -> Rec:
    S1, per, lim, _ = geometry(n)
    if k == 5:                                             # an A-run of 17: starts p, p + 1
        s = _bg(rng, n)
        p = int(rng.integers(n))
        _put(s, p, b"A" * 17)
        return _finish(s, [p, (p + 1) % n], 3, k, reverse)
    r32, r2 = (lambda: int(rng.integers(32))), (lambda: int(rng.integers(2)))    # noqa: E731
    sd = int(reverse)

    def draw():
        if k == 0:                                         # same step, same strand (only locate's popcount sees it)
            t = int(rng.integers(S1))
            return [(sd, t, r32(), KEY), (sd, t, r32(), KEY)]
        if k == 1:                                         # same step, opposite strands
            t = int(rng.integers(S1))
            return [(0, t, r32(), KEY), (1, t, r32(), KEY)]
        if k == 2:                                         # same lane, different steps
            t = int(rng.integers(lane_steps(n, 0)[1]))
            return [(r2(), t, r32(), KEY), (r2(), t + 1, r32(), KEY)]
        if k == 3:                                         # different lanes
            ln = 1 + int(rng.integers(used_lanes(n) - 1))
            return [(r2(), int(rng.integers(4 * per)), r32(), KEY), (r2(), lane_steps(n, ln)[r2()], r32(), KEY)]
        s2 = r2()                                          # one in S1, one in the last full step
        return [(s2, S1, _s1_rotation(rng, n, s2), KEY), (r2(), S1 - 1, r32(), KEY)]
    return _in_steps(rng, n, draw, 3, k, reverse)


def three_or_more(rng, n: int, m: int) -> Rec:
    gap = n // m
    plants = []
    for i in range(m):
        w = i * gap + int(rng.integers(0, gap - 40))
        plants.append((i & 1, w if i & 1 == 0 else (n - 16 - w) % n, KEY))
    return _planted(rng, n, plants, 4, m, bool(rng.integers(2)))


# ---------------------------------------------------------------- the corpus
def corpus(seed: int = 5) -> list[Rec]:
    rng = np.random.default_rng(seed)
    out = []
    for i, n in enumerate(LENGTHS):
        out += [one_key(rng, n, sd, p) for p in sweep_starts(n, rng) for sd in (0, 1)]
        out += [one_key(rng, n, 1, p) for p in reverse_sweep(n, rng)]
        reps = 2 if n in FULL_SWEEP else 1
        out += [near_miss(rng, n, k, bool((i + k + r) & 1)) for k in range(4) for r in range(reps)]
        out += [two_keys(rng, n, k, bool((i + k + r) & 1)) for k in range(6) for r in range(reps)]
        out.append(three_or_more(rng, n, 3 + i % 3))
        out.append(Rec(structured(rng, n, i).seq, 5))
    return out


# ---------------------------------------------------------------- brute force (CPU)
def keys(s: bytes) -> np.ndarray:
    """the 16-mer key (2 bits per base, first base in the top bits) of every rotation of s"""
    c = _CODE[np.frombuffer(s, np.uint8)].astype(np.uint32)
    c = np.concatenate([c, c[:15]])
    k = np.zeros(len(s), dtype=np.uint32)
    for i in range(16):
        k = (k << np.uint32(2)) | c[i: i + len(s)]
    return k


def occurrences(s: bytes, value: int = 0):
    """[(strand, start)] of every rotation of either strand whose 16-mer key is `value`"""
    return [(sd, int(p)) for sd, x in ((0, s), (1, revcomp(s))) for p in np.flatnonzero(keys(x) == value)]


NEAR_VALUE = 1                                             # A x 15 C


def min_key_occurrences(s: bytes):
    ks = [keys(s), keys(revcomp(s))]
    m = int(min(ks[0].min(), ks[1].min()))
    return m, [(sd, int(p)) for sd in (0, 1) for p in np.flatnonzero(ks[sd] == m)]
