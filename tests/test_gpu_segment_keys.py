"""The segment kernel (k_canon_seg, ck_seg2.cuh: one warp per 2-bit record of 8 193 .. 425 984 bases, a lane per segment) on
records whose minimal 16-mer sits on purpose at its scan-lane, step, partial-step, wrap and 1024-base block boundaries
(tests/seg_key_corpus.py), against the oracle: canonical bytes, lengths, (start, strand), XXH3-64 and first indices must be
identical.

The kernel runs on batches in the doubled packed2 layout with aligned output (or none): the host-buffer entries (ASCII and
host-packed), ck_dev_canon_bytes, ck_dev_canon_packed2 and the FASTA text entry.  Same-offsets output and a context created
under CK_SEG_KERNEL=0 send the same records to k_canon_cta<2>, which is checked too.  Records whose minimal 16-mer occurs more
than once go to k_canon_cta<2>'s duel path: the retry counts per family show that the kernel finishes every other record
itself and retries each tie exactly once."""
import numpy as np
import pytest

import lane_tie_corpus as L
import oracle
import seg_key_corpus as S
from oracle import cli as ocli
from test_gpu_lane_ties import Corpus, _compare

pytestmark = pytest.mark.gpu

CLS_C2A, CLS_C2B = 2, 3                                      # ck_kernels.cuh: n <= 65 536, n <= 425 984


@pytest.fixture(scope="module")
def seg():
    return Corpus(S.corpus())


@pytest.fixture(scope="module")
def short(seg):
    """the records up to 33 793 bases, and every eighth longer one: what the uniq and FASTA text tests take"""
    return seg.subset([i for i, r in enumerate(seg.recs) if len(r.seq) <= 33793 or i % 8 == 0])


def _context(**kw):
    import circkit_b200
    return circkit_b200.Context(**{"max_batch_bytes": 128 << 20, "max_batch_records": 1 << 14, "table_capacity": 1 << 15, **kw})


@pytest.fixture(scope="module")
def ctx():
    c = _context()
    yield c
    c.close()


@pytest.fixture(scope="module")
def ctx_generic():
    """long 2-bit records to the CTA kernels only (the variable is read when the context is created)"""
    with pytest.MonkeyPatch.context() as mp:
        mp.setenv("CK_SEG_KERNEL", "0")
        c = _context()
    yield c
    c.close()


def _counts(ws):
    # the workspace begins with the run's counters: u32 32 + c counts the records a kernel appended to class c's retry list
    c = ws.buf[:256].cpu().numpy().view(np.uint32)
    return int(c[32 + CLS_C2A]), int(c[32 + CLS_C2B])


def _bytes_run(ctx, c, want_bytes=True, want_hash=True):
    """ck_dev_canon_bytes -> (results as numpy, retries (C2A, C2B), kernel times)"""
    import torch
    from circkit_b200 import device as D
    dev = torch.device("cuda", ctx.device)
    n, total = len(c.seqs), int(c.off[-1])
    raw = torch.from_numpy(c.arena.copy()).to(dev)
    outs = D.CanonOutputs(n, total, dev, want_bytes=want_bytes, want_hash=want_hash, aligned=True)
    lens = torch.empty(n, dtype=torch.int32, device=dev)
    ws = D.Workspace(ctx, n, total)
    ctx._lib.ck_kernel_timing(ctx.handle, 1)
    D.kernel_times(ctx)
    D.canon_bytes(ctx, raw, torch.from_numpy(c.off.astype(np.int64)).to(dev), n, total, outs, lens, ws, normalize=False)
    D.check(ctx, ws)
    times = D.kernel_times(ctx)
    ctx._lib.ck_kernel_timing(ctx.handle, 0)
    got = dict(lens=lens.cpu().numpy(), start=outs.start.cpu().numpy(), strand=outs.strand.cpu().numpy(),
               hash=None if outs.hash is None else outs.hash.cpu().numpy(), out=None if outs.out is None else outs.out.cpu().numpy())
    return got, _counts(ws), times


# ---------------------------------------------------------------- host entries
@pytest.mark.parametrize("aligned,no_bytes", [(True, False), (True, True), (False, False)],
                         ids=["aligned", "aligned-no-bytes", "same-offsets"])
def test_host_canonicalize(ctx, seg, aligned, no_bytes):
    got = ctx.canonicalize_batch(seg.arena, seg.off, normalize=False, want_bytes=not no_bytes, aligned=aligned)
    _compare(seg, got, aligned, f"aligned={aligned} no_bytes={no_bytes}")


def test_host_packed(ctx, seg):
    got = ctx.canonicalize_batch_packed(seg.arena, seg.off, normalize=False, aligned=True, threads=8)
    _compare(seg, got, True, "host-packed")


# ---------------------------------------------------------------- device entries
@pytest.mark.parametrize("want_bytes,want_hash", [(False, False), (False, True), (True, False), (True, True)])
def test_device_bytes_entry(ctx, seg, want_bytes, want_hash):
    got, _, times = _bytes_run(ctx, seg, want_bytes, want_hash)
    assert times["2bit_seg_8193_425984"][1] == 1, times
    _compare(seg, got, True, f"ck_dev_canon_bytes bytes={want_bytes} hash={want_hash}")


@pytest.mark.parametrize("mode", ["list", "two-class"])
def test_device_packed2_entry(ctx, seg, mode):
    """ck_dev_canon_packed2 on the doubled arena packed by lane_tie_corpus.pack2: list mode, and the promise CLS_C2A | CLS_C2B"""
    import torch
    from circkit_b200 import device as D
    dev = torch.device("cuda", ctx.device)
    off, words = L.pack2(seg.seqs, False)
    b = D.DeviceBatch(torch.from_numpy(off.astype(np.int64)).to(dev), torch.from_numpy(words.view(np.int64)).to(dev), len(seg.seqs),
                      int(off[-1]), False)
    del words
    outs = D.CanonOutputs(b.n, b.total, dev, aligned=True)
    ws = D.Workspace(ctx, b.n)
    ctx._lib.ck_kernel_timing(ctx.handle, 1)
    D.kernel_times(ctx)
    D.canon_packed2(ctx, b, outs, ws, class_mask=0 if mode == "list" else (1 << CLS_C2A) | (1 << CLS_C2B))
    D.check(ctx, ws)
    times = D.kernel_times(ctx)
    ctx._lib.ck_kernel_timing(ctx.handle, 0)
    assert times["2bit_seg_8193_425984"][1] == 1, times
    got = dict(start=outs.start.cpu().numpy(), strand=outs.strand.cpu().numpy(), hash=outs.hash.cpu().numpy(),
               out=outs.out.cpu().numpy())
    _compare(seg, got, True, f"ck_dev_canon_packed2 {mode}")


def test_cta_kernels_on_the_same_records(ctx_generic, seg):
    got = ctx_generic.canonicalize_batch(seg.arena, seg.off, aligned=True)
    _compare(seg, got, True, "CK_SEG_KERNEL=0 host")
    dgot, retried, times = _bytes_run(ctx_generic, seg)
    assert times["2bit_seg_8193_425984"][1] == 0 and retried == (0, 0), times
    _compare(seg, dgot, True, "CK_SEG_KERNEL=0 device")


# ---------------------------------------------------------------- uniq and the FASTA text entry
def test_uniq_two_slots_survivors(ctx, short):
    """rotations and reverse complements (some starting inside the key's A-run) collapse onto their first occurrence across
    two batches on the two slots, ASCII and host-packed; the survivors come back with their canonical bytes"""
    from circkit_b200 import core
    seqs = L.rotations_and_revcomps(short.seqs, np.random.default_rng(31))
    c = Corpus([L.Rec(s, -1) for s in seqs])
    wh, wfirst = oracle.uniq_consume(c.want["out"], c.off, c.want["lens"])
    assert (wfirst != np.arange(len(seqs))).sum() > 0.2 * len(short.seqs)
    keep = np.flatnonzero(wfirst == np.arange(len(seqs), dtype=np.uint64))
    cut = len(seqs) // 2
    for packed in (False, True):
        ctx.uniq_reset()
        got_idx = []
        for k, (lo, hi) in enumerate([(0, cut), (cut, len(seqs))]):
            o = c.off[lo: hi + 1] - c.off[lo]
            a = np.ascontiguousarray(c.arena[int(c.off[lo]): int(c.off[hi])])
            if packed:
                ctx.uniq_submit_packed(k, core.pack2_host(a, o, threads=8), lo, aligned=True, survivors=True)
            else:
                ctx.uniq_submit(k, a, o, lo, normalize=False, aligned=True, survivors=True)
            r = ctx.uniq_wait_survivors(k, hi - lo, int(o[-1]))
            assert np.array_equal(r["first"], wfirst[lo:hi]) and np.array_equal(r["hash"], wh[lo:hi]), packed
            for j, i in enumerate(r["index"]):
                g, c0 = lo + int(i), int(r["offsets"][j])
                got_idx.append(g)
                assert r["bytes"][c0: c0 + int(c.lens[g])].tobytes() == c.want["out"][int(c.off[g]): int(c.off[g + 1])].tobytes(), g
        assert got_idx == [int(x) for x in keep], packed
    ctx.uniq_reset()


def test_fasta_text(ctx, short):
    """ck_fasta_submit: canonicalize, uniq and uniq -c, lines wrapped at 80 (every other record unwrapped), byte for byte
    against the oracle's restatement of the CLI"""
    def wrap(s, w):
        return b"\n".join(s[i: i + w] for i in range(0, len(s), w)) if w else s
    text = b"".join(b">r%d f%d\n%s\n" % (i, r.family, wrap(r.seq, 80 * (i % 2))) for i, r in enumerate(short.recs))
    assert ctx.fasta_submit(0, text, "canonicalize") == len(short.recs)
    assert ctx.fasta_wait(0)["fasta"] == ocli.cli_canonicalize(text, threads=8)
    dups = L.rotations_and_revcomps(short.seqs[::2], np.random.default_rng(32))
    text = b"".join(b">d%d\n%s\n" % (i, wrap(s, 61 * (i % 2))) for i, s in enumerate(dups))
    for slot, canonical in ((1, False), (0, True)):
        ctx.uniq_reset()
        assert ctx.fasta_submit(slot, text, "uniq", canonical_body=canonical) == len(dups)
        assert ctx.fasta_wait(slot)["fasta"] == ocli.cli_uniq(text, canonicalize=canonical, threads=8)[0], canonical
    ctx.uniq_reset()


# ---------------------------------------------------------------- k_canon_seg does its share
@pytest.mark.parametrize("want_hash", [False, True], ids=["no-hash", "hash"])
def test_segment_kernel_does_its_share(ctx, seg, want_hash):
    """One family per batch through ck_dev_canon_bytes.  k_canon_seg finishes every record whose minimal 16-mer occurs once
    (one key, near miss) itself, and sends every record whose minimal 16-mer occurs twice or more -- in one step, one lane or
    two lanes, on one strand or both -- to CLS_C2A (n <= 65 536) or CLS_C2B, exactly once"""
    fams = {}
    for i, r in enumerate(seg.recs):
        fams.setdefault(r.family, []).append(i)
    for fam, ix in sorted(fams.items()):
        batch = seg.subset(ix)
        got, retried, times = _bytes_run(ctx, batch, True, want_hash)
        assert times["2bit_seg_8193_425984"][1] == 1, times
        _compare(batch, got, True, f"hash={want_hash} family {fam}")
        ties = [r.family in S.TIE_FAMILIES or (r.family == 5 and len(S.min_key_occurrences(r.seq)[1]) > 1) for r in batch.recs]
        want = (sum(t and len(r.seq) <= 65536 for t, r in zip(ties, batch.recs)), sum(t and len(r.seq) > 65536 for t, r in zip(ties, batch.recs)))
        print(f"retries: k_canon_seg hash={want_hash} family={fam} records={len(batch.recs)} retried(C2A, C2B)={retried} "
              f"expected={want}")
        assert retried == want, (fam, len(batch.recs), retried, want)
