"""Records built on purpose for the tie logic of the 2-bit lane kernels (ck_stream2.cuh, ck_stream3.cuh), and a numpy packer for
both packed2 arena layouts (ck_device.cuh).  Helper of tests/test_lane_tie_corpus.py and tests/test_gpu_lane_ties.py; it holds
no tests.

"Key" below is the minimal 8-mer over both strands and all rotations of a record.  Every family plants AAAAAAAA, the smallest
8-mer there is, into a background that cannot make it: the background is over {C, G, T}, and every 4th base (and base 0) is not
T, so that no T-run is longer than 5 even across the record end -- the reverse strand then has no A-run of 8 either.  A planted
key is followed by a 16-base continuation drawn the same way (bases 8 .. 23 of its rotation, what the lane kernel compares to
tell two occurrences apart, s3_ext16).

An occurrence is (strand, start) in the strand's own coordinates: strand 0 is the record, strand 1 its reverse complement.  The
lane kernel scans a record in steps of 32 rotations; `kernel_step` restates which step sees an occurrence.  A reverse-strand
record of any family is the reverse complement of a forward construction: its occurrences keep their starts and flip strand.

Families (`Rec.family`):
  0  random over ACGT;
  1  one key (`occ` has one entry), its forward window swept over every residue mod 32 and over n - 8 .. n - 1 (wrapping);
  2  two keys on the same strand whose continuations first differ at base k < 16 (`k`), same 32-rotation step or not;
  3  two keys on opposite strands, k < 16;
  4  two keys whose continuations agree for 16 bases or more (k = 16): planted, a dimer h + h, a circle h + revcomp(h);
  5  three or more keys;
  6  two keys (either strand pairing), the continuation of one wraps the record end, k < 16;
  7  structure: homopolymer, cut power, near-periodic, long A-run, dimer, reverse-palindromic circle, trimer.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

A8 = b"AAAAAAAA"
_COMP = bytes.maketrans(b"ACGT", b"TGCA")
_CODE = np.full(256, 255, dtype=np.uint8)
_CODE[list(b"ACGT")] = [0, 1, 2, 3]

SINGLE_LENGTHS = list(range(1, 513))
DOUBLED_LENGTHS = [513, 1023, 1024, 1025, 1100, 2047, 2048, 2049, 4095, 4096, 4097, 8191, 8192]
# distances between the two keys of a pair (same strand): 1 = an A-run of 9, 9 .. 23 = the first continuation runs into the
# second key, >= 24 = disjoint; below 32 the pair can share a step
PAIR_D = [1, 9, 12, 16, 20, 23, 24, 25, 27, 31, 32, 33, 40, 63, 64, 100]
# forward key position minus reverse key window (opposite strands): >= 9 or <= -40 keeps the two blocks disjoint
OPP_D = [9, 10, 16, 23, 24, 31, 32, 33, 40, 64, 100, -40, -41, -47, -63, -64, -100]


@dataclass
class Rec:
    seq: bytes
    family: int
    occ: tuple = ()          # ((strand, start), ...) of the key, where declared
    k: int | None = None     # pairs: first continuation base that differs (16: the first 16 agree)


def revcomp(s: bytes) -> bytes:
    return s.translate(_COMP)[::-1]


def kernel_step(n: int, strand: int, start: int) -> int:
    """The lane kernel's scan step that sees occurrence (strand, start): forward start p in step p >> 5; a reverse-strand start
    covers forward window f = n - 8 - start, seen by step t for f in 32 t + 9 .. 32 t + 40 (windows 0 .. 8 by the last step)."""
    if strand == 0:
        return start >> 5
    f = (n - 8 - start) % n
    return ((f if f >= 9 else f + n) - 9) >> 5


def _bg(rng, n: int) -> bytearray:
    """n bases over {C, G, T}; base 0 and every 4th base are C or G"""
    s = rng.choice(np.frombuffer(b"CGT", np.uint8), n)
    s[3::4] = rng.choice(np.frombuffer(b"CG", np.uint8), len(s[3::4]))
    if n:
        s[0] = rng.choice(np.frombuffer(b"CG", np.uint8))
    return bytearray(s.tobytes())


def _cont_pair(rng, k: int, length: int = 16):
    """two continuations (drawn like the background) whose first difference is at base k (k >= length: identical)"""
    c1 = _bg(rng, length)
    c2 = _bg(rng, length)
    c2[:min(k, length)] = c1[:min(k, length)]
    if k < length:
        opts = [b for b in (b"CG" if (k % 4 == 3 or k == 0) else b"CGT") if b != c1[k]]
        c2[k] = opts[int(rng.integers(len(opts)))]
    return bytes(c1), bytes(c2)


def _put(s: bytearray, pos: int, data: bytes):
    n = len(s)
    for i, b in enumerate(data):
        s[(pos + i) % n] = b


def _finish(s: bytearray, occ_fwd, family: int, k, reverse: bool) -> Rec:
    """occ_fwd: key starts planted on the forward strand of s (and reverse ones, as (strand, start))"""
    occ = tuple(sorted(o if isinstance(o, tuple) else (0, o) for o in occ_fwd))
    if reverse:
        return Rec(revcomp(bytes(s)), family, tuple(sorted((1 - sd, st) for sd, st in occ)), k)
    return Rec(bytes(s), family, occ, k)


def _window_to_start(n: int, strand: int, w: int) -> int:
    """start, in strand coordinates, of the key whose forward window begins at w"""
    return w % n if strand == 0 else (n - 8 - w) % n


# ---------------------------------------------------------------- families
def unique_key(rng, n: int, w: int, strand: int) -> Rec:
    """family 1: one key; its forward window starts at w (n >= 9)"""
    s = _bg(rng, n)
    p = _window_to_start(n, strand, w)
    _put(s, p, A8 + bytes(_bg(rng, 16))[: max(0, min(16, n - 9))])
    return _finish(s, [p], 1, None, strand == 1)


def _pair_block(rng, d: int, k: int, tail: int = 16):
    """forward block with keys at 0 and d, continuations that first differ at base k (k = 16: the first `tail` bases of the two
    continuations agree, then they differ unless tail == 16).  Returns (block, k as the block really has it)."""
    c1, c2 = _cont_pair(rng, k, tail)
    if d == 1:                                             # an A-run of 9: continuations A + c2 and c2 differ at base 0
        return A8 + b"A" + c2, 0
    if d < 24:                                             # the first continuation runs into the second key (base d - 8 is A)
        return A8 + c1[: d - 8] + A8 + c2, min(k, d - 8)
    return A8 + c1 + bytes(_bg(rng, d - 8 - len(c1))) + A8 + c2, k


def pair_same_strand(rng, n: int, w1: int, d: int, k: int, strand: int, family: int = 2, tail: int = 16) -> Rec:
    """families 2 / 4 / 6: keys with forward windows w1 and w1 + d on one strand (n >= d + 40)"""
    s = _bg(rng, n)
    blk, k = _pair_block(rng, d, k, tail)
    if strand == 0:
        p1 = w1 % n
    else:                                                  # windows w1, w1 + d of the record = starts q + d, q of the builder
        p1 = (n - 8 - w1 - d) % n
    _put(s, p1, blk)
    return _finish(s, [p1, (p1 + d) % n], family, k, strand == 1)


def pair_opposite(rng, n: int, w: int, d: int, k: int, flip: bool, family: int = 3, tail: int = 16) -> Rec:
    """families 3 / 4 / 6: a forward key at window w + d, a reverse-strand key at window w (blocks disjoint: d >= 9 or d <= -40)"""
    s = _bg(rng, n)
    c1, c2 = _cont_pair(rng, k, tail)
    f = w % n
    p = (w + d) % n
    _put(s, f - 16, revcomp(A8 + c2[:16]) + b"C")        # T8 at f .. f + 7, then a base that is not T
    _put(s, p, A8 + c1)
    return _finish(s, [p, (1, (n - 8 - f) % n)], family, min(k, 16), flip)


def three_or_more(rng, n: int, m: int, shape: int) -> Rec:
    """family 5: m >= 3 keys: m separate blocks (mixing strands), or an A-run of m + 7 (shape 1)"""
    s = _bg(rng, n)
    if shape == 1 or n // m < 32:
        p = int(rng.integers(n))
        _put(s, p, b"A" * (m + 7))
        return _finish(s, [(p + i) % n for i in range(m)], 5, None, bool(rng.integers(2)))
    gap = n // m
    occ = []
    for i in range(m):
        base = i * gap + int(rng.integers(0, max(1, gap - 30)))
        c = bytes(_bg(rng, 16))
        if i % 2 and shape == 2:                           # a reverse-strand key
            _put(s, base, revcomp(A8 + c) + b"C")
            occ.append((1, (n - 8 - (base + 16)) % n))
        else:
            _put(s, base, A8 + c)
            occ.append(base % n)
    return _finish(s, occ, 5, None, bool(rng.integers(2)))


def full_tie(rng, n: int, palindrome: bool) -> Rec:
    """family 4, n even: h + h or h + revcomp(h) with one key in h"""
    h = n // 2
    u = unique_key(rng, h, int(rng.integers(h - 8)), 0)     # the key does not wrap h: it stays whole in h + revcomp(h)
    p = u.occ[0][1]
    if palindrome:
        # revcomp(h) holds the key on the reverse strand of the circle: reverse start = p (the circle is its own reverse complement)
        return Rec(u.seq + revcomp(u.seq), 4, tuple(sorted([(0, p), (1, p)])), 16)
    return Rec(u.seq + u.seq, 4, ((0, p), (0, p + h)), 16)


def _rand(rng, n: int, alpha: bytes = b"ACGT") -> bytes:
    return rng.choice(np.frombuffer(alpha, np.uint8), n).astype(np.uint8).tobytes()


def structured(rng, n: int, kind: int) -> Rec:
    """family 7: the shapes of test_gpu_parity._with_structure"""
    kind %= 7
    if kind == 0:
        s = bytes([b"ACGT"[int(rng.integers(4))]]) * n                        # homopolymer
    elif kind == 1:
        u = _rand(rng, int(rng.integers(1, max(2, min(40, n) + 1))))
        s = (u * (n // len(u) + 1))[:n]                                        # cut power
    elif kind == 2:
        u = _rand(rng, int(rng.integers(1, 6)))
        b = bytearray((u * (n // len(u) + 1))[:n])
        for _ in range(int(rng.integers(0, 3))):
            b[int(rng.integers(n))] = b"ACGT"[int(rng.integers(4))]           # near-periodic
        s = bytes(b)
    elif kind == 3:
        b = bytearray(_rand(rng, n))
        a, L = int(rng.integers(n)), int(rng.integers(1, n + 1))
        for i in range(L):
            b[(a + i) % n] = ord("A")                                         # long A-run
        s = bytes(b)
    elif kind == 4 and n % 2 == 0:
        h = _rand(rng, n // 2); s = h + h                                      # dimer
    elif kind == 5 and n % 2 == 0:
        h = _rand(rng, n // 2); s = h + revcomp(h)                             # reverse-palindromic circle
    elif kind == 6 and n % 3 == 0:
        h = _rand(rng, n // 3); s = h * 3                                      # trimer
    else:
        s = (b"ACGT"[int(rng.integers(4)):] + b"ACGT" * (n // 4 + 1))[:n]
    return Rec(s, 7)


# ---------------------------------------------------------------- corpora
def _pair_window(rng, n: int, d: int, strand: int, same_step: bool) -> int:
    """forward window of the first key of a same-strand pair: both in one step (d < 32) or not"""
    r = int(rng.integers(0, 32 - d)) if same_step and d < 32 else int(rng.integers(max(0, 32 - d), 32)) if d < 32 else int(rng.integers(32))
    j = int(rng.integers(0, max(1, (n - d - 40) // 32)))
    return 32 * j + r + (9 if strand else 0)


def _length_records(rng, n: int, i: int, full: bool) -> list[Rec]:
    """the records of length n; i cycles the sweeps; full: every (window, strand) of family 1 and every k of the pairs"""
    recs = [Rec(_rand(rng, n), 0), structured(rng, n, i)]
    if n >= 9:
        wins = sorted(set(list(range(min(32, n))) + list(range(max(0, n - 8), n))))
        if full:
            recs += [unique_key(rng, n, w, sd) for w in wins for sd in (0, 1)]
        else:
            recs += [unique_key(rng, n, wins[i % len(wins)], 0), unique_key(rng, n, wins[(i + 17) % len(wins)], 1)]
    if n < 96:
        return recs
    pd = [x for x in PAIR_D if x + 40 <= n]
    od = [x for x in OPP_D if abs(x) + 40 <= n]
    for r in range(16 if full else 1):
        j, k = i + 5 * r, (i + r) % 16
        for sd in (0, 1):                                  # family 2, both strands, the keys in two steps
            d = pd[(j // 2 + 3 * sd) % len(pd)]
            recs.append(pair_same_strand(rng, n, _pair_window(rng, n, d, sd, False), d, k, sd))
        for sd in ((0, 1) if full else ((i >> 4) & 1,)):  # family 2 in one step with every k: disjoint keys 24 .. 31 apart
            d = (24, 25, 27, 31)[j % 4]
            recs.append(pair_same_strand(rng, n, _pair_window(rng, n, d, sd, True), d, k, sd))
        recs.append(pair_opposite(rng, n, int(rng.integers(n)), od[j % len(od)], (k + 7) % 16, bool(j % 2)))   # family 3
        # family 6: the continuation of one key wraps the record end (its start in n - 23 .. n - 9)
        st = n - 23 + (j % 15)
        if j % 3 == 2:
            recs.append(pair_opposite(rng, n, st - 40, 40, k, False, family=6))
        elif j % 3 == 1:
            recs.append(pair_same_strand(rng, n, st, 40, k, 0, family=6))
        else:
            recs.append(pair_same_strand(rng, n, (n - 48 - st) % n, 40, k, 1, family=6))
    # family 4: continuations that agree for 16 bases or more; full ties
    tail = 16 + (i % 9 if n >= 100 else 0)                # continuations agree for `tail` bases, then differ
    recs.append(pair_same_strand(rng, n, int(rng.integers(n)), 40, 16, i % 2, family=4, tail=tail))
    recs.append(pair_opposite(rng, n, int(rng.integers(n)), 40, 16, bool(i % 2), family=4, tail=tail))
    if n % 2 == 0:
        recs.append(full_tie(rng, n, bool((i // 2) % 2)))
    recs.append(three_or_more(rng, n, 3 + i % 3, i % 3))                                                          # family 5
    return recs


def single_copy_corpus(seed: int = 1) -> list[Rec]:
    """every length 1 .. 512 (the single-copy arena): families where they fit, random and structured records otherwise"""
    rng = np.random.default_rng(seed)
    out = []
    for n in SINGLE_LENGTHS:
        out += _length_records(rng, n, n, False)
    return out


def doubled_corpus(seed: int = 2) -> list[Rec]:
    """boundary lengths of the doubled arena's lane classes (513 .. 8192)"""
    rng = np.random.default_rng(seed)
    out = []
    for i, n in enumerate(DOUBLED_LENGTHS):
        out += _length_records(rng, n, i, True)
    return out


def rotations_and_revcomps(seqs: list[bytes], rng, run: bytes = b"AAAA") -> list[bytes]:
    """seqs, followed by duplicates that must collapse onto them: rotations (half of them starting inside the run of the key,
    i.e. inside a tie; `run` finds it), reverse complements, and both"""
    out = list(seqs)
    for s in seqs:
        n = len(s)
        if not n or rng.random() < 0.5:
            continue
        a = s.find(run)
        r = (a + int(rng.integers(0, 8))) % n if a >= 0 and rng.random() < 0.5 else int(rng.integers(n))
        t = s[r:] + s[:r]
        out.append(revcomp(t) if rng.random() < 0.5 else t)
    perm = rng.permutation(len(out) - len(seqs)) + len(seqs)
    return out[: len(seqs)] + [out[i] for i in perm]


# ---------------------------------------------------------------- brute force (CPU)
def _codes(s: bytes) -> np.ndarray:
    return _CODE[np.frombuffer(s, np.uint8)].astype(np.int64)


def rotation_windows(s: bytes, start: np.ndarray, length: int) -> np.ndarray:
    """bases start .. start + length - 1 (mod n) of s as 2-bit codes, one row per start"""
    c = _codes(s)
    idx = (start[:, None] + np.arange(length)[None, :]) % len(s)
    return c[idx]


def key_occurrences(s: bytes):
    """(key as int, [(strand, start)] of every rotation of either strand that begins with it), over all 2 n rotations"""
    n = len(s)
    w = 4 ** np.arange(7, -1, -1, dtype=np.int64)
    keys = [rotation_windows(x, np.arange(n), 8) @ w for x in (s, revcomp(s))]
    key = int(min(keys[0].min(), keys[1].min()))
    occ = [(sd, int(p)) for sd in (0, 1) for p in np.flatnonzero(keys[sd] == key)]
    return key, occ


def continuation(s: bytes, strand: int, start: int) -> np.ndarray:
    """bases 8 .. 23 of the rotation (strand, start)"""
    x = s if strand == 0 else revcomp(s)
    return rotation_windows(x, np.array([start]), 24)[0, 8:]


def first_difference(s: bytes, a, b) -> int:
    """first base (0 .. 15) at which the continuations of occurrences a and b differ; 16 if they agree"""
    d = np.flatnonzero(continuation(s, *a) != continuation(s, *b))
    return int(d[0]) if d.size else 16


# ---------------------------------------------------------------- packed2 arenas
def pack2(seqs: list[bytes], single: bool):
    """-> (offsets uint64[n + 1], arena uint64 words) in the packed2 layout of ck_device.cuh.  single-copy: record i at 16-byte
    granule (offsets[i] >> 6) + 2 i, units 0 .. (n >> 4) + 4; doubled: 32-byte granule (offsets[i] >> 6) + 3 i, units
    0 .. max((2 n + 143) >> 4, (n >> 4) + 5).  A unit is a u32 of 16 bases, first base in the high bits, unit j holds
    S[b mod n]; whatever else the arena holds is zero."""
    lens = np.array([len(s) for s in seqs], dtype=np.uint64)
    off = np.zeros(len(seqs) + 1, dtype=np.uint64)
    np.cumsum(lens, out=off[1:])
    total, nrec = int(off[-1]), len(seqs)
    words = 2 * ((total >> 6) + 2 * nrec + 2) if single else 4 * ((total >> 6) + 3 * nrec + 3)
    units = np.zeros(2 * words, dtype=np.uint32)
    wts = np.uint64(4) ** np.arange(15, -1, -1, dtype=np.uint64)
    for s, (u0, nu) in zip(seqs, unit_ranges(lens, single)):
        if not s:
            continue
        c = _codes(s).astype(np.uint64)[np.arange(16 * nu) % len(s)].reshape(nu, 16)
        units[u0: u0 + nu] = (c * wts).sum(axis=1).astype(np.uint32)
    return off, units.view(np.uint64)


def unit_ranges(lens, single: bool):
    """(first u32 index, unit count) of every record's defined units in a pack2 arena"""
    off = np.concatenate([[0], np.cumsum(np.asarray(lens, dtype=np.int64))])
    out = []
    for i, n in enumerate(lens):
        n, o = int(n), int(off[i])
        out.append((4 * ((o >> 6) + 2 * i), (n >> 4) + 5) if single else (8 * ((o >> 6) + 3 * i), max((2 * n + 143) >> 4, (n >> 4) + 5) + 1))
    return out
