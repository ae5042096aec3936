"""Records over {-, A, C, G, N, T} built on purpose for the 4-bit lane kernel (k_pack4 + k_canon_l4, ck_lane4.cuh).  Helper of
tests/test_key_corpora.py and tests/test_gpu_lane4_keys.py; it holds no tests.

The kernel's keys are 8-mers of 4-bit codes (- A C G N T = 0 .. 5).  Every family plants KEY = "-------A" into a background
over {A, C, G, N, T}: no background window starts with '-', and a window that starts inside a planted run is larger than KEY.
The base in front of a planted run of '-' is never T -- the reverse strand would read "-------" + complement(T) = KEY there
(`_plant` writes that guard base).  '-' and N complement to themselves.

An occurrence is (strand, start) in the strand's own coordinates: strand 0 is the record, strand 1 its reverse complement.
k_pack4 stores both strands as arrays of their own, so the scan sees occurrence (strand, start) in oct start >> 6, unit
start >> 3 of that strand's array; the partial oct J1 = n >> 6 holds rotations 64 J1 .. n - 1.  A reverse-strand record of
a family is the reverse complement of a forward construction: its occurrences keep their starts and flip strand.

Families (`Rec.family`):
  1  one key; its start swept over every residue mod 64, every unit and oct edge, n - 8 .. n - 1 (wrapping), the last
     rotation of the partial oct and rotation 0 (the first one past its mask), both strands;
  2  one key and the near miss NEAR = "-------C": `k` 0 same oct, 1 another oct, 2 the near miss on the opposite strand;
  3  two keys: `k` 0 opposite strands, starts in the same unit; 1 same strand, same oct; 2 same strand, different octs;
     3 opposite strands, different octs; 4 "T-------A" (the two occurrences overlap); 5 one key in the partial oct, one in
     the last full oct; 6 one key wrapping the record end, one in oct 0;
  4  a self-complementary minimal key: `k` 0 "--------", 1 "---NN---" (flanked "A---NN---T"): one run, both strands;
  5  three or more keys;
  6  structure: homopolymers of '-' and N, cut powers, dimers, reverse-palindromic circles, random (`occ` not declared);
  7  one key at the class edges 128, 129, 240, 241, 2048, 2049 (lane tag, hash limit, class limit);
  8  the mixed batch (`mixed_batch`): one-key records of the lane's lengths, paired in input order with a record the
     lane cannot take -- `k` 0 an IUPAC letter (library semantics), 1 shorter than 129, 2 longer than 2048.
"""
from __future__ import annotations

import numpy as np

from lane_tie_corpus import Rec, _finish, _put, revcomp

KEY = b"-------A"
NEAR = b"-------C"
ALPHA = b"-ACGNT"
IUPAC = b"RYKMSWBDHV"
_CODE = np.full(256, 255, dtype=np.uint8)
_CODE[list(ALPHA)] = range(6)

SWEEP_LENGTHS = list(range(129, 193)) + [240, 241, 255, 256, 257, 319, 320, 321, 447, 448, 449, 511, 512, 513, 1023, 1024,
                                         1025, 2047, 2048]
EDGE_LENGTHS = [128, 129, 240, 241, 2048, 2049]
TIE_FAMILIES = (3, 4, 5)


def _bg(rng, n: int) -> bytearray:
    return bytearray(rng.choice(np.frombuffer(b"ACGNT", np.uint8), n).tobytes())


def _rand(rng, n: int, alpha: bytes = ALPHA) -> bytes:
    return rng.choice(np.frombuffer(alpha, np.uint8), n).astype(np.uint8).tobytes()


def footprint(n: int, strand: int, start: int, length: int = 8) -> set:
    """forward positions a planted word and its guard base occupy"""
    if strand == 0:
        return {(start - 1 + i) % n for i in range(length + 1)}
    f = (n - length - start) % n
    return {(f + i) % n for i in range(length + 1)}


def _plant(rng, s: bytearray, strand: int, start: int, word: bytes):
    """word at (strand, start); the base in front of it on its strand becomes A, C or N: not T (the reverse strand would read
    KEY there) nor G (it would read NEAR there)"""
    n, g = len(s), b"ACN"[int(rng.integers(3))]
    if strand == 0:
        _put(s, start, word)
        s[(start - 1) % n] = g
    else:
        f = (n - len(word) - start) % n
        _put(s, f, revcomp(word))
        s[(f + len(word)) % n] = revcomp(bytes([g]))[0]    # g in front of the word on strand 1


def _planted(rng, n: int, plants, family: int, k=None, reverse: bool = False) -> Rec:
    """plants: [(strand, start, word)] with disjoint footprints; occ = the plants of the smallest word"""
    used = set()
    for sd, st, w in plants:
        fp = footprint(n, sd, st, len(w))
        assert not fp & used, (n, plants)
        used |= fp
    s = _bg(rng, n)
    for sd, st, w in plants:
        _plant(rng, s, sd, st, w)
    m = min(w for _, _, w in plants)
    return _finish(s, [(sd, st) for sd, st, w in plants if w == m], family, k, reverse)


def _free(rng, n: int, taken, strand: int, lo: int = 0, hi: int | None = None) -> int:
    """a start in [lo, hi) whose footprint misses every forward position in `taken`"""
    hi = n if hi is None else hi
    for _ in range(1000):
        st = int(rng.integers(lo, hi))
        if not footprint(n, strand, st) & taken:
            return st
    raise AssertionError((n, lo, hi))


def one_key(rng, n: int, start: int, strand: int, family: int = 1) -> Rec:
    return _planted(rng, n, [(0, start, KEY)], family, None, strand == 1)


def sweep_starts(n: int, i: int) -> list[int]:
    """family 1's starts at length n: every residue mod 64 (in an oct that moves with i), every unit edge of one full oct, every
    oct edge, n - 8 .. n - 1, the last rotation of the partial oct and rotation 0"""
    octs = (n + 63) >> 6
    st = set()
    for r in range(64):
        p = 64 * ((r + i) % octs) + r
        st.add(p if p < n else r)
    st |= {64 * (i % (n >> 6)) + 8 * u + e for u in range(8) for e in (0, 7)}
    st |= {(64 * j + e) % n for j in range(1, octs + 1) for e in (-1, 0)}
    st |= set(range(n - 8, n)) | {0, n - 1}
    return sorted(st)


def near_miss(rng, n: int, k: int, reverse: bool) -> Rec:
    octs = n >> 6
    if k < 2:
        o1 = int(rng.integers(octs))
        a = 64 * o1 + int(rng.integers(0, 54))
        if k == 0:
            b = a + int(rng.integers(10, 64 - (a & 63))) if (a & 63) < 54 else a - 10
        else:
            o2 = (o1 + 1 + int(rng.integers(octs - 1))) % octs
            b = _free(rng, n, footprint(n, 0, a), 0, 64 * o2, min(64 * o2 + 64, n))
        plants = [(0, a, KEY), (0, b, NEAR)]
    else:
        a = int(rng.integers(n))
        plants = [(0, a, KEY), (1, _free(rng, n, footprint(n, 0, a), 1), NEAR)]
    return _planted(rng, n, plants, 2, k, reverse)


def two_keys(rng, n: int, k: int, reverse: bool) -> Rec:
    octs, J1 = (n + 63) >> 6, n >> 6
    if k == 0:                                             # opposite strands, starts in the same unit
        for _ in range(1000):
            a = int(rng.integers(n - 8))
            b = 8 * (a >> 3) + int(rng.integers(8))
            if b < n and not footprint(n, 0, a) & footprint(n, 1, b):
                return _planted(rng, n, [(0, a, KEY), (1, b, KEY)], 3, k, reverse)
        raise AssertionError(n)
    if k == 1:                                             # same strand, same oct, different units
        o = int(rng.integers(J1))
        a = 64 * o + int(rng.integers(0, 40))
        b = a + int(rng.integers(10, 64 - (a & 63)))
        return _planted(rng, n, [(0, a, KEY), (0, b, KEY)], 3, k, reverse)
    if k == 2:                                             # same strand, different octs
        a = int(rng.integers(n))
        b = _free(rng, n, footprint(n, 0, a), 0)
        while (a >> 6) == (b >> 6):
            b = _free(rng, n, footprint(n, 0, a), 0)
        return _planted(rng, n, [(0, a, KEY), (0, b, KEY)], 3, k, reverse)
    if k == 3:                                             # opposite strands, different octs
        a = int(rng.integers(n))
        b = _free(rng, n, footprint(n, 0, a), 1)
        while (a >> 6) == (b >> 6):
            b = _free(rng, n, footprint(n, 0, a), 1)
        return _planted(rng, n, [(0, a, KEY), (1, b, KEY)], 3, k, reverse)
    if k == 4:                                             # "T-------A": KEY at p, and the reverse strand's KEY at n - 7 - p
        s = _bg(rng, n)
        p = int(rng.integers(n))
        _put(s, p - 1, b"T" + KEY)
        return _finish(s, [(0, p), (1, (n - 7 - p) % n)], 3, k, reverse)
    if k == 5 and n & 63 >= 10:                            # the partial oct and the last full oct
        a = 64 * J1 + int(rng.integers(1, n & 63))
        b = _free(rng, n, footprint(n, 0, a), 0, 64 * (J1 - 1), 64 * J1)
        return _planted(rng, n, [(0, a, KEY), (0, b, KEY)], 3, k, reverse)
    a = n - 1 - int(rng.integers(7))                       # k 6 (and 5 where the partial oct is short): KEY wraps the end
    b = _free(rng, n, footprint(n, 0, a), 0, 0, 64)
    return _planted(rng, n, [(0, a, KEY), (0, b, KEY)], 3, 6, reverse)


def self_complementary(rng, n: int, k: int) -> Rec:
    s = _bg(rng, n)
    p = int(rng.integers(n))
    if k == 0:
        _put(s, p, b"--------")
    else:
        _put(s, p - 1, b"A---NN---T")
    return Rec(bytes(s), 4, tuple(sorted([(0, p), (1, (n - 8 - p) % n)])), k)


def three_or_more(rng, n: int, m: int) -> Rec:
    gap = n // m
    plants = [(i & 1 if m > 3 else 0, i * gap + int(rng.integers(0, gap - 20)), KEY) for i in range(m)]
    plants = [(sd, st if sd == 0 else (n - 8 - st) % n, w) for sd, st, w in plants]
    return _planted(rng, n, plants, 5, m, bool(rng.integers(2)))


def structured(rng, n: int, kind: int) -> Rec:
    kind %= 7
    if kind == 0:
        s = b"-" * n
    elif kind == 1:
        s = b"N" * n
    elif kind == 2:
        u = _rand(rng, int(rng.integers(1, 41)))
        s = (u * (n // len(u) + 1))[:n]                                        # cut power
    elif kind == 3 and n % 2 == 0:
        h = _rand(rng, n // 2); s = h + h                                      # dimer
    elif kind == 4 and n % 2 == 0:
        h = _rand(rng, n // 2); s = h + revcomp(h)                             # reverse-palindromic circle
    elif kind == 5:
        s = bytes(b"-N"[int(x)] for x in rng.integers(0, 2, n))                # the two self-complementary symbols
    else:
        s = _rand(rng, n)
    return Rec(s, 6)


# ---------------------------------------------------------------- corpora
def corpus(seed: int = 3) -> list[Rec]:
    rng = np.random.default_rng(seed)
    out = []
    for i, n in enumerate(SWEEP_LENGTHS):
        out += [one_key(rng, n, p, sd) for p in sweep_starts(n, i) for sd in (0, 1)]
        out += [near_miss(rng, n, k, bool((i + k) & 1)) for k in range(3)]
        out += [two_keys(rng, n, k, bool((i + k) & 1)) for k in range(7)]
        out += [self_complementary(rng, n, i & 1), three_or_more(rng, n, 3 + i % 3)]
        out += [structured(rng, n, i + j) for j in range(2)]
    for n in EDGE_LENGTHS:
        out += [one_key(rng, n, p, sd, family=7) for p in (0, 7, 8, 63, 64, n // 2, n - 8, n - 1) for sd in (0, 1)]
    return out


def mixed_batch(seed: int = 4) -> list[Rec]:
    """family 8: (lane record, other record) pairs, in either order within the pair (= the two halves of a k_pack4 warp); the
    lane records' byte offsets take every residue mod 32"""
    rng = np.random.default_rng(seed)
    out, off, ctl = [], 0, 0
    for i in range(192):
        n = SWEEP_LENGTHS[(7 * i) % len(SWEEP_LENGTHS)]
        e = one_key(rng, n, int(rng.integers(n)), i & 1, family=8)
        k = i % 3
        first = (i >> 2) & 1                               # 1: the other record is the first of the pair
        if k == 0:                                         # same length, one IUPAC letter
            s = bytearray(_rand(rng, n, b"ACGNT"))
            s[int(rng.integers(n))] = IUPAC[int(rng.integers(len(IUPAC)))]
            x = Rec(bytes(s), 8, (), 0)
        else:                                              # < 129 or > 2048, of a length that puts the lane record after it
            base = 97 if k == 1 else 2049                  # at the next residue mod 32
            m = base + (ctl - off - base) % 32 if first else base + int(rng.integers(32))
            ctl += first
            x = Rec(_rand(rng, m), 8, (), k)
        pair = [x, e] if first else [e, x]
        out += pair
        off += len(pair[0].seq) + len(pair[1].seq)
    return out


def cli_spelling(seq: bytes, rng) -> bytes:
    """seq as a FASTA body may spell it for `normalize=True`: '-' as '.' or '~' (or itself), N as an IUPAC letter, lower case,
    U for T, and '\\r', ' ', '\\t' inside the record"""
    out = bytearray()
    r = rng.random(len(seq))
    c = rng.integers(0, 1 << 16, len(seq))
    for b, x, y in zip(seq, r, c):
        if b == 45:
            ch = b"-.~"[y % 3]
        elif b == 78:
            ch = (IUPAC + b"N")[y % 11]
        elif b == 84 and x < 0.3:
            ch = 85
        else:
            ch = b
        if 65 <= ch <= 90 and (y >> 8) & 1:
            ch += 32
        out.append(ch)
        if x > 0.97:
            out += b"\r \t"[y % 3: y % 3 + 1]
    return bytes(out)


def rotations_and_revcomps(seqs: list[bytes], rng) -> list[bytes]:
    """lane_tie_corpus.rotations_and_revcomps with the rotations that start inside a run of '-'"""
    import lane_tie_corpus
    return lane_tie_corpus.rotations_and_revcomps(seqs, rng, run=b"----")


# ---------------------------------------------------------------- brute force (CPU)
def codes(s: bytes) -> np.ndarray:
    return _CODE[np.frombuffer(s, np.uint8)].astype(np.int64)


def keys(s: bytes) -> np.ndarray:
    """the 8-mer key (4-bit codes, first symbol in the top nibble) of every rotation of s"""
    c = codes(s)
    n = len(c)
    idx = (np.arange(n)[:, None] + np.arange(8)[None, :]) % n
    return c[idx] @ (16 ** np.arange(7, -1, -1, dtype=np.int64))


def key_value(w: bytes) -> int:
    return int(codes(w) @ (16 ** np.arange(7, -1, -1, dtype=np.int64)))


def key_occurrences(s: bytes):
    """(minimal key, [(strand, start)] of every rotation of either strand that begins with it), over all 2 n rotations"""
    ks = [keys(s), keys(revcomp(s))]
    key = int(min(ks[0].min(), ks[1].min()))
    return key, [(sd, int(p)) for sd in (0, 1) for p in np.flatnonzero(ks[sd] == key)]


def word_occurrences(s: bytes, w: bytes):
    v = key_value(w)
    return [(sd, int(p)) for sd, x in ((0, s), (1, revcomp(s))) for p in np.flatnonzero(keys(x) == v)]


def lane_retries(n: int, ties: bool, want_hash: bool) -> bool:
    """whether k_canon_l4 sends a {-ACGNT} record to the retry list: below its length limits, or the minimal key occurs twice"""
    return n <= 2048 and (n < (241 if want_hash else 129) or ties)
