"""The 4-bit lane kernel (k_pack4 + k_canon_l4, ck_lane4.cuh) on records whose minimal 8-mer sits on purpose at its oct, unit,
partial-oct, wrap and strand boundaries (tests/lane4_key_corpus.py), against the oracle: canonical bytes, lengths, (start,
strand), XXH3-64 and first indices must be identical.

The kernel runs where a batch has a packed4 arena and aligned output (or none): the host-buffer entries, ck_dev_canon_bytes and
the FASTA text entry.  Same-offsets output and a context created under CK_L4_KERNEL=0 send the same records to the generic
kernels, which are checked too.  A kernel that skipped a rotation at a boundary gets these records wrong; one that saw a
rotation twice only sends them to k_canon_warp<4> -- the retry counts per family show that."""
import numpy as np
import pytest

import lane4_key_corpus as Q
import oracle
from oracle import cli as ocli
from test_gpu_lane_ties import Corpus, _compare

pytestmark = pytest.mark.gpu

CLS_W4 = 4                                                   # ck_kernels.cuh


@pytest.fixture(scope="module")
def keys():
    return Corpus(Q.corpus())


@pytest.fixture(scope="module")
def mixed():
    return Corpus(Q.mixed_batch())


def _context(**kw):
    import circkit_b200
    return circkit_b200.Context(**{"max_batch_bytes": 32 << 20, "max_batch_records": 1 << 16, "table_capacity": 1 << 17, **kw})


@pytest.fixture(scope="module")
def ctx():
    c = _context()
    yield c
    c.close()


@pytest.fixture(scope="module")
def ctx_generic():
    """{-ACGNT} records to the generic 4-bit kernels only (the variable is read when the context is created)"""
    with pytest.MonkeyPatch.context() as mp:
        mp.setenv("CK_L4_KERNEL", "0")
        c = _context()
    yield c
    c.close()


def _device_run(ctx, c, want_bytes=True, want_hash=True, normalize=False, seqs=None):
    """ck_dev_canon_bytes over c (or over `seqs`, spellings of c's records) -> (results as numpy, k_canon_l4's retries, kernel
    times)"""
    import torch
    from circkit_b200 import device as D
    dev = torch.device("cuda", ctx.device)
    seqs = c.seqs if seqs is None else seqs
    off = np.zeros(len(seqs) + 1, dtype=np.int64)
    np.cumsum([len(s) for s in seqs], out=off[1:])
    n, total = len(seqs), int(off[-1])
    raw = torch.from_numpy(np.frombuffer(b"".join(seqs), dtype=np.uint8).copy()).to(dev)
    outs = D.CanonOutputs(n, total, dev, want_bytes=want_bytes, want_hash=want_hash, aligned=True)
    lens = torch.empty(n, dtype=torch.int32, device=dev)
    ws = D.Workspace(ctx, n, total)
    ctx._lib.ck_kernel_timing(ctx.handle, 1)
    D.kernel_times(ctx)
    D.canon_bytes(ctx, raw, torch.from_numpy(off).to(dev), n, total, outs, lens, ws, normalize=normalize)
    D.check(ctx, ws)
    times = D.kernel_times(ctx)
    ctx._lib.ck_kernel_timing(ctx.handle, 0)
    # the workspace begins with the run's counters: u32 32 + c counts the records a kernel appended to class c's retry list
    counts = ws.buf[:256].cpu().numpy().view(np.uint32)
    got = dict(lens=lens.cpu().numpy(), start=outs.start.cpu().numpy(), strand=outs.strand.cpu().numpy(),
               hash=None if outs.hash is None else outs.hash.cpu().numpy(), out=None if outs.out is None else outs.out.cpu().numpy())
    return got, int(counts[32 + CLS_W4]), times


# ---------------------------------------------------------------- host entries
@pytest.mark.parametrize("aligned,no_bytes", [(True, False), (True, True), (False, False)],
                         ids=["aligned", "aligned-no-bytes", "same-offsets"])
@pytest.mark.parametrize("batch", ["keys", "mixed"])
def test_host_canonicalize(ctx, keys, mixed, batch, aligned, no_bytes):
    c = keys if batch == "keys" else mixed
    got = ctx.canonicalize_batch(c.arena, c.off, normalize=False, want_bytes=not no_bytes, aligned=aligned)
    _compare(c, got, aligned, f"{batch} aligned={aligned} no_bytes={no_bytes}")


def test_cli_spelling(ctx, keys):
    """CLI semantics ('-' as '.' / '~', N as IUPAC letters, lower case, U, whitespace inside the record) give the plain
    records' results: in the oracle, through the host entry and through ck_dev_canon_bytes (normalised lengths differ from the
    offset spans)"""
    rng = np.random.default_rng(21)
    spelled = [Q.cli_spelling(s, rng) for s in keys.seqs]
    assert sum(len(a) != len(b) for a, b in zip(spelled, keys.seqs)) > len(spelled) // 4
    arena = np.frombuffer(b"".join(spelled), dtype=np.uint8)
    off = np.zeros(len(spelled) + 1, dtype=np.uint64)
    np.cumsum([len(s) for s in spelled], out=off[1:])
    want = oracle.canonicalize_batch(arena, off, normalize=True, threads=8)
    assert np.array_equal(want["lens"], keys.want["lens"])
    for k in ("start", "strand", "hash"):
        assert np.array_equal(want[k], keys.want[k]), k
    got = ctx.canonicalize_batch(arena, off, normalize=True, aligned=True)
    assert np.array_equal(got["lens"], keys.want["lens"])
    for k in ("start", "strand", "hash"):
        assert np.array_equal(got[k], keys.want[k]), k
    starts = ctx.aligned_starts(off).astype(np.int64)
    for i in range(len(spelled)):
        a, m = int(keys.off[i]), int(keys.lens[i])
        assert got["out"][starts[i]: starts[i] + m].tobytes() == keys.want["out"][a: a + m].tobytes(), (i, keys.recs[i].family)
    dgot, _, times = _device_run(ctx, keys, normalize=True, seqs=spelled)
    assert times["4bit_lane_129_2048"][1] == 1, times
    out = dgot.pop("out")
    _compare(keys, dgot, True, "ck_dev_canon_bytes cli spelling")
    for i in range(len(spelled)):                          # aligned slots at the spelled offsets, normalised lengths
        a, m = int(keys.off[i]), int(keys.lens[i])
        assert out[starts[i]: starts[i] + m].tobytes() == keys.want["out"][a: a + m].tobytes(), (i, keys.recs[i].family)


# ---------------------------------------------------------------- ck_dev_canon_bytes
@pytest.mark.parametrize("want_bytes,want_hash", [(False, False), (False, True), (True, False), (True, True)])
@pytest.mark.parametrize("batch", ["keys", "mixed"])
def test_device_entry(ctx, keys, mixed, batch, want_bytes, want_hash):
    c = keys if batch == "keys" else mixed
    got, _, times = _device_run(ctx, c, want_bytes, want_hash)
    assert times["4bit_lane_129_2048"][1] == 1 and times["pack4"][1] == 1, times
    _compare(c, got, True, f"{batch} bytes={want_bytes} hash={want_hash}")


def test_generic_kernels_on_the_same_records(ctx_generic, keys, mixed):
    for c in (keys, mixed):
        got = ctx_generic.canonicalize_batch(c.arena, c.off, aligned=True)
        _compare(c, got, True, "CK_L4_KERNEL=0 host")
        dgot, retried, times = _device_run(ctx_generic, c)
        assert times["4bit_lane_129_2048"][1] == 0 and retried == 0, times
        _compare(c, dgot, True, "CK_L4_KERNEL=0 device")


# ---------------------------------------------------------------- uniq and the FASTA text entry
def test_uniq_two_slots_survivors(ctx, keys):
    """rotations and reverse complements (some starting inside the run of '-') collapse onto their first occurrence across two
    batches on the two slots; the survivors come back with their canonical bytes"""
    seqs = Q.rotations_and_revcomps(keys.seqs, np.random.default_rng(22))
    c = Corpus([Q.Rec(s, -1) for s in seqs])
    wh, wfirst = oracle.uniq_consume(c.want["out"], c.off, c.want["lens"])
    assert (wfirst != np.arange(len(seqs))).sum() > 0.2 * len(keys.seqs)
    keep = np.flatnonzero(wfirst == np.arange(len(seqs), dtype=np.uint64))
    cut = len(seqs) // 2
    ctx.uniq_reset()
    got_idx, got_bytes = [], []
    for k, (lo, hi) in enumerate([(0, cut), (cut, len(seqs))]):
        o = c.off[lo: hi + 1] - c.off[lo]
        ctx.uniq_submit(k, np.ascontiguousarray(c.arena[int(c.off[lo]): int(c.off[hi])]), o, lo, normalize=False, aligned=True,
                        survivors=True)
        r = ctx.uniq_wait_survivors(k, hi - lo, int(o[-1]))
        assert np.array_equal(r["first"], wfirst[lo:hi]) and np.array_equal(r["hash"], wh[lo:hi])
        for j, i in enumerate(r["index"]):
            g, c0 = lo + int(i), int(r["offsets"][j])
            got_idx.append(g)
            got_bytes.append(r["bytes"][c0: c0 + int(c.lens[g])].tobytes())
    ctx.uniq_reset()
    assert got_idx == [int(x) for x in keep]
    for g, b in zip(got_idx, got_bytes):
        assert b == c.want["out"][int(c.off[g]): int(c.off[g + 1])].tobytes(), g


def _wrap(s: bytes, width: int) -> bytes:
    return b"\n".join(s[i: i + width] for i in range(0, len(s), width)) if width else s


@pytest.mark.parametrize("spelling", ["plain", "cli"])
def test_fasta_text(ctx, keys, spelling):
    """ck_fasta_submit: canonicalize, uniq and uniq -c, lines wrapped at 60 (every third record unwrapped), byte for byte
    against the oracle's restatement of the CLI"""
    rng = np.random.default_rng(23)
    seqs = keys.seqs if spelling == "plain" else [Q.cli_spelling(s, rng) for s in keys.seqs]
    text = b"".join(b">r%d f%d\n%s\n" % (i, r.family, _wrap(s, 60 * (i % 3 != 0))) for i, (r, s) in enumerate(zip(keys.recs, seqs)))
    assert ctx.fasta_submit(0, text, "canonicalize") == len(seqs)
    assert ctx.fasta_wait(0)["fasta"] == ocli.cli_canonicalize(text, threads=8)
    dups = Q.rotations_and_revcomps(keys.seqs, np.random.default_rng(24))
    if spelling == "cli":
        dups = [Q.cli_spelling(s, rng) for s in dups]
    text = b"".join(b">d%d\n%s\n" % (i, _wrap(s, 70 * (i % 2))) for i, s in enumerate(dups))
    for slot, canonical in ((1, False), (0, True)):
        ctx.uniq_reset()
        assert ctx.fasta_submit(slot, text, "uniq", canonical_body=canonical) == len(dups)
        assert ctx.fasta_wait(slot)["fasta"] == ocli.cli_uniq(text, canonicalize=canonical, threads=8)[0], canonical
    ctx.uniq_reset()


# ---------------------------------------------------------------- k_canon_l4 does its share
def _expected_retries(c, i, want_hash):
    r = c.recs[i]
    n = len(r.seq)
    if r.family == 8 and not r.occ:                       # the other record of a mixed pair: IUPAC or < 129 retried, > 2048 not
        return n <= 2048
    if set(r.seq) <= set(b"ACGT"):                         # a structured record without '-' or N: the 2-bit lane's
        return False
    ties = r.family in Q.TIE_FAMILIES or (r.family == 6 and len(Q.key_occurrences(r.seq)[1]) > 1)
    return Q.lane_retries(n, ties, want_hash)


@pytest.mark.parametrize("want_hash", [False, True], ids=["no-hash", "hash"])
def test_lane_kernel_does_its_share(ctx, keys, mixed, want_hash):
    """One family per batch through ck_dev_canon_bytes.  k_canon_l4 finishes a record whose minimal key occurs once itself (from
    129 symbols, 241 with a hash); every record whose key occurs twice or more (on one strand or on both), every record below
    those lengths and every record with another symbol goes to k_canon_warp<4>, exactly once"""
    fams = {}
    for i, r in enumerate(keys.recs):
        fams.setdefault((r.family, "short" if len(r.seq) < 241 else "long"), []).append(i)
    batches = [(f, keys.subset(ix)) for f, ix in sorted(fams.items())] + [((8, "mixed"), mixed)]
    for fam, batch in batches:
        got, retried, times = _device_run(ctx, batch, True, want_hash)
        assert times["4bit_lane_129_2048"][1] == 1 and times["pack4"][1] == 1, times
        _compare(batch, got, True, f"hash={want_hash} family {fam}")
        want = sum(_expected_retries(batch, i, want_hash) for i in range(len(batch.recs)))
        print(f"retries: k_canon_l4 hash={want_hash} family={fam[0]} lengths={fam[1]} records={len(batch.recs)} "
              f"retried={retried} expected={want}")
        assert retried == want, (fam, len(batch.recs), retried, want)
