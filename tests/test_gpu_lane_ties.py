"""The 2-bit lane kernels on records built for their tie logic (tests/lane_tie_corpus.py), against the oracle: canonical bytes,
lengths, (start, strand), XXH3-64 and first indices must be identical.

Batches whose records are all <= 512 bases use the single-copy packed2 arena and k_canon_s2 (plus k_canon_w2 for the retries and
the same-offsets output); longer batches use the doubled arena and k_canon_s3, or k_canon_s2 in a context created under
CK_LANE_KERNEL=2.  Every path is run: the host entries, the FASTA text entry, uniq over two slots, ck_dev_canon_packed2 on arenas
packed here in either layout (list mode, direct mode, a two-class promise, every bytes / hash variant), and the lane kernel's
retry counts per family -- the results stay right if the lane kernel sends its ties to the retry kernels, so only the counts show
that it resolves them itself."""
import numpy as np
import pytest

import lane_tie_corpus as L
import oracle
from oracle import cli as ocli

pytestmark = pytest.mark.gpu

CLS_W2S, CLS_W2M, CLS_W2L, CLS_W2X = 0, 1, 10, 11            # ck_kernels.cuh
LANE_CLASSES = (CLS_W2S, CLS_W2M, CLS_W2L, CLS_W2X)


class Corpus:
    def __init__(self, recs):
        self.recs = recs
        self.seqs = [r.seq for r in recs]
        self.lens = np.array([len(s) for s in self.seqs], dtype=np.int64)
        self.off = np.zeros(len(recs) + 1, dtype=np.uint64)
        np.cumsum(self.lens, out=self.off[1:])
        self.arena = np.frombuffer(b"".join(self.seqs), dtype=np.uint8)
        self.want = oracle.canonicalize_batch(self.arena, self.off, normalize=False, threads=8)

    def subset(self, keep):
        return Corpus([self.recs[i] for i in keep])


@pytest.fixture(scope="module")
def single():
    return Corpus(L.single_copy_corpus())


@pytest.fixture(scope="module")
def doubled():
    return Corpus(L.doubled_corpus())


def _context(**kw):
    import circkit_b200
    return circkit_b200.Context(**{"max_batch_bytes": 64 << 20, "max_batch_records": 1 << 16, "table_capacity": 1 << 16, **kw})


@pytest.fixture(scope="module")
def ctx():
    c = _context()
    yield c
    c.close()


@pytest.fixture(scope="module")
def ctx_s2():
    """k_canon_s2 for the doubled arena too (the variable is read when the context is created)"""
    with pytest.MonkeyPatch.context() as mp:
        mp.setenv("CK_LANE_KERNEL", "2")
        c = _context()
    yield c
    c.close()


def _gather(out, off, aligned):
    """canonical bytes of every record, back in the compact layout"""
    lens = (off[1:] - off[:-1]).astype(np.int64)
    total = int(off[-1])
    if not aligned:
        return out[:total]
    starts = (32 * ((off[:-1] >> np.uint64(5)) + np.arange(len(lens), dtype=np.uint64))).astype(np.int64)
    return out[np.repeat(starts - off[:-1].astype(np.int64), lens) + np.arange(total, dtype=np.int64)]


def _compare(c, got, aligned=True, tag=""):
    """got: dict of numpy arrays (lens, start, strand, hash, out -- each optional)"""
    want = c.want
    n = len(c.recs)
    bad = np.zeros(n, dtype=bool)
    if got.get("lens") is not None:
        bad |= got["lens"][:n].astype(np.int64) != want["lens"].astype(np.int64)
    if got.get("start") is not None:
        bad |= (got["start"][:n].astype(np.uint32) != want["start"]) | (got["strand"][:n] != want["strand"])
    if got.get("hash") is not None:
        bad |= got["hash"][:n].view(np.uint64) != want["hash"]
    if got.get("out") is not None:
        diff = np.flatnonzero(_gather(got["out"], c.off, aligned) != want["out"][: int(c.off[-1])])
        bad[np.searchsorted(c.off[1:], diff.astype(np.uint64), side="right")] = True
    idx = np.flatnonzero(bad)
    rep = [(int(i), c.recs[i].family, int(c.lens[i]), c.recs[i].occ, c.recs[i].k, int(want["start"][i]), int(want["strand"][i]),
            None if got.get("start") is None else (int(got["start"][i]), int(got["strand"][i]))) for i in idx[:4]]
    assert idx.size == 0, f"{tag}: {idx.size} records differ from the oracle, first (index, family, n, occ, k, want, got): {rep}"


# ---------------------------------------------------------------- a. host entries on single-copy batches
@pytest.mark.parametrize("aligned", [False, True], ids=["same-offsets", "aligned"])
@pytest.mark.parametrize("no_bytes", [False, True], ids=["bytes", "no-bytes"])
def test_host_canonicalize(ctx, single, aligned, no_bytes):
    got = ctx.canonicalize_batch(single.arena, single.off, normalize=False, want_bytes=not no_bytes, aligned=aligned)
    _compare(single, got, aligned, f"aligned={aligned} no_bytes={no_bytes}")


@pytest.mark.parametrize("normalize", [False, True], ids=["lib", "cli"])
def test_host_normalize(ctx, single, normalize):
    """CLI semantics on lower-case and RNA spellings of the same records give the same results as the records themselves"""
    seqs = single.seqs
    if normalize:
        seqs = [s.lower() if i % 4 == 1 else s.replace(b"T", b"U") if i % 4 == 2 else s.lower().replace(b"t", b"u") if i % 4 == 3
                else s for i, s in enumerate(seqs)]
    arena = np.frombuffer(b"".join(seqs), dtype=np.uint8)
    want = oracle.canonicalize_batch(arena, single.off, normalize=normalize, threads=8)
    for k in ("lens", "start", "strand", "hash", "out"):
        assert np.array_equal(want[k], single.want[k]), k
    got = ctx.canonicalize_batch(arena, single.off, normalize=normalize, aligned=True)
    _compare(single, got, True, f"normalize={normalize}")


@pytest.mark.parametrize("aligned", [False, True], ids=["same-offsets", "aligned"])
def test_host_packed(ctx, single, aligned):
    got = ctx.canonicalize_batch_packed(single.arena, single.off, normalize=False, aligned=aligned, threads=4)
    _compare(single, got, aligned, f"packed aligned={aligned}")


@pytest.mark.parametrize("packed", [False, True], ids=["ascii-in", "packed-in"])
def test_uniq_two_slots_survivors(ctx, single, packed):
    """rotations and reverse complements (some starting inside the key's run) collapse onto their first occurrence, across two
    batches on the two slots, and the survivors come back with their canonical bytes"""
    from circkit_b200 import core
    seqs = L.rotations_and_revcomps(single.seqs, np.random.default_rng(8))
    c = Corpus([L.Rec(s, -1) for s in seqs])
    wh, wfirst = oracle.uniq_consume(c.want["out"], c.off, c.want["lens"])
    assert (wfirst != np.arange(len(seqs))).sum() > 0.2 * len(single.seqs)
    keep = np.flatnonzero(wfirst == np.arange(len(seqs), dtype=np.uint64))
    cut = len(seqs) // 2
    ctx.uniq_reset()
    got_idx, got_bytes = [], []
    for k, (lo, hi) in enumerate([(0, cut), (cut, len(seqs))]):
        o = c.off[lo: hi + 1] - c.off[lo]
        a = np.ascontiguousarray(c.arena[int(c.off[lo]): int(c.off[hi])])
        if packed:
            pb = core.pack2_host(a, o, normalize=True, threads=2)
            ctx.uniq_submit_packed(k, pb, lo, aligned=True, survivors=True)
        else:
            ctx.uniq_submit(k, a, o, lo, normalize=True, aligned=True, survivors=True)
        r = ctx.uniq_wait_survivors(k, hi - lo, int(o[-1]))
        assert np.array_equal(r["first"], wfirst[lo:hi]) and np.array_equal(r["hash"], wh[lo:hi])
        assert np.array_equal(r["lens"], c.want["lens"][lo:hi])
        for j, i in enumerate(r["index"]):
            g, c0 = lo + int(i), int(r["offsets"][j])
            got_idx.append(g)
            got_bytes.append(r["bytes"][c0: c0 + int(c.lens[g])].tobytes())
    ctx.uniq_reset()
    assert got_idx == [int(x) for x in keep]
    for g, b in zip(got_idx, got_bytes):
        assert b == c.want["out"][int(c.off[g]): int(c.off[g + 1])].tobytes(), g


def test_fasta_text(ctx, single):
    """ck_fasta_submit: canonicalize, uniq and uniq -c on a one-line-per-record FASTA of the corpus (with duplicates), byte for
    byte against the oracle's restatement of the CLI"""
    text = b"".join(b">r%d f%d\n%s\n" % (i, r.family, r.seq) for i, r in enumerate(single.recs))
    assert ctx.fasta_submit(0, text, "canonicalize") == len(single.recs)
    assert ctx.fasta_wait(0)["fasta"] == ocli.cli_canonicalize(text, threads=8)
    dups = L.rotations_and_revcomps(single.seqs, np.random.default_rng(9))
    text = b"".join(b">d%d\n%s\n" % (i, s) for i, s in enumerate(dups))
    for slot, canonical in ((1, False), (0, True)):
        ctx.uniq_reset()
        assert ctx.fasta_submit(slot, text, "uniq", canonical_body=canonical) == len(dups)
        assert ctx.fasta_wait(slot)["fasta"] == ocli.cli_uniq(text, canonicalize=canonical, threads=8)[0], canonical
    ctx.uniq_reset()


# ---------------------------------------------------------------- b. layout invariance
@pytest.mark.parametrize("aligned", [False, True], ids=["same-offsets", "aligned"])
def test_one_long_record_switches_the_layout_not_the_results(ctx, single, aligned):
    """a 513-base record moves the whole batch to the doubled arena (k_canon_s3): the other records' outputs do not change"""
    extra = L.unique_key(np.random.default_rng(4), 513, 8, 1).seq
    arena = np.concatenate([single.arena, np.frombuffer(extra, np.uint8)])
    off = np.concatenate([single.off, [single.off[-1] + np.uint64(513)]])
    a = ctx.canonicalize_batch(single.arena, single.off, aligned=aligned)
    b = ctx.canonicalize_batch(arena, off, aligned=aligned)
    n = len(single.recs)
    for k in ("lens", "start", "strand", "hash"):
        assert np.array_equal(a[k], b[k][:n]), k
    assert np.array_equal(_gather(a["out"], single.off, aligned), _gather(b["out"], off, aligned)[: int(single.off[-1])])
    assert b["out"][(int(ctx.aligned_starts(off)[n]) if aligned else int(single.off[-1])):][:513].tobytes() == oracle.canonicalize(extra)


# ---------------------------------------------------------------- c. the device entry on arenas packed here
def _device_run(ctx, c, single_layout, want_bytes=True, want_hash=True, class_mask=0, timing=False):
    """ck_dev_canon_packed2 over c packed by lane_tie_corpus.pack2 -> (results as numpy, retry counts per class, kernel times)"""
    import torch
    from circkit_b200 import device as D
    dev = torch.device("cuda", ctx.device)
    off, words = L.pack2(c.seqs, single_layout)
    b = D.DeviceBatch(torch.from_numpy(off.astype(np.int64)).to(dev), torch.from_numpy(words.view(np.int64)).to(dev), len(c.seqs),
                      int(off[-1]), single_layout)
    n = len(c.seqs)
    outs = D.CanonOutputs(n, b.total, dev, want_bytes=want_bytes, want_hash=want_hash, aligned=True)
    ws = D.Workspace(ctx, n)
    if timing:
        ctx._lib.ck_kernel_timing(ctx.handle, 1)
        D.kernel_times(ctx)
    D.canon_packed2(ctx, b, outs, ws, class_mask=class_mask)
    D.check(ctx, ws)
    times = None
    if timing:
        times = D.kernel_times(ctx)
        ctx._lib.ck_kernel_timing(ctx.handle, 0)
    # ws.buf begins with the run's 64 u32 counters (ck_lib.cu:385, a.retry_counts = io.counts + 32): u32 32 + c counts the
    # records the lane kernel appended to the retry list of class c (ck_stream2.cuh / ck_stream3.cuh, end of the record loop)
    counts = ws.buf[:256].cpu().numpy().view(np.uint32)
    got = dict(start=outs.start.cpu().numpy(), strand=outs.strand.cpu().numpy(),
               hash=None if outs.hash is None else outs.hash.cpu().numpy(), out=None if outs.out is None else outs.out.cpu().numpy())
    return got, {cl: int(counts[32 + cl]) for cl in LANE_CLASSES}, times


@pytest.mark.parametrize("single_layout", [True, False], ids=["single-copy", "doubled"])
def test_pack2_reproduces_the_synthetic_arena(ctx, single_layout):
    """the packer of lane_tie_corpus writes the words ck_synth_packed2 writes for the same records (every defined unit)"""
    from circkit_b200 import device as D
    b = D.synth_batch(ctx, seed=7, first_index=0, n_records=400, kind=0, lo=1, hi=512 if single_layout else 3000,
                      dup_permille=200, single=single_layout)
    ascii_ = D.unpack_ascii(ctx, b).cpu().numpy()
    off = b.offsets.cpu().numpy().astype(np.uint64)
    seqs = [ascii_[int(off[i]): int(off[i + 1])].tobytes() for i in range(400)]
    poff, words = L.pack2(seqs, single_layout)
    assert np.array_equal(poff, off)
    got, mine = b.packed2.cpu().numpy().view(np.uint32), words.view(np.uint32)
    for i, (u0, nu) in enumerate(L.unit_ranges([len(s) for s in seqs], single_layout)):
        assert np.array_equal(got[u0: u0 + nu], mine[u0: u0 + nu]), (i, len(seqs[i]))


@pytest.mark.parametrize("mode", ["list", "direct", "two-class"])
@pytest.mark.parametrize("want_bytes,want_hash", [(False, False), (False, True), (True, False), (True, True)])
@pytest.mark.parametrize("single_layout", [True, False], ids=["single-copy", "doubled"])
def test_device_entry(ctx, single, single_layout, want_bytes, want_hash, mode):
    mask = {"list": 0, "direct": 1 << CLS_W2S, "two-class": (1 << CLS_W2S) | (1 << CLS_W2M)}[mode]
    got, _, _ = _device_run(ctx, single, single_layout, want_bytes, want_hash, mask)
    _compare(single, got, True, f"single_layout={single_layout} bytes={want_bytes} hash={want_hash} {mode}")


# ---------------------------------------------------------------- d. the lane kernel resolves its share of the ties
def _family_batches(c, min_n=0):
    fams = {}
    for i, r in enumerate(c.recs):
        if r.family in (1, 2, 3, 6) and len(r.seq) < max(129, min_n):
            continue                                          # below 129 bases every record is the retry kernels' (hash: n <= 128)
        fams.setdefault(r.family, []).append(i)
    return {f: c.subset(ix) for f, ix in sorted(fams.items())}


@pytest.mark.parametrize("want_hash", [False, True], ids=["no-hash", "hash"])
@pytest.mark.parametrize("kernel", ["s2-single", "s3-doubled", "s2-doubled"])
def test_lane_kernel_does_its_share(ctx, ctx_s2, single, doubled, kernel, want_hash):
    """One family per batch.  The lane kernel finishes a record with one key itself; two keys whose continuations differ in the
    first 16 bases are told apart in the lane (k_canon_s3 always, k_canon_s2 in the variants without a hash: ck_stream2.cuh,
    kPair); two keys that agree for 16 bases, and three or more keys, always go to the retry list."""
    c2 = ctx_s2 if kernel == "s2-doubled" else ctx
    single_layout = kernel == "s2-single"
    pair_in_lane = not (kernel.startswith("s2") and want_hash)
    corpora = [single] if single_layout else [single, doubled]
    for c in corpora:
        for fam, batch in _family_batches(c).items():
            got, retry, times = _device_run(c2, batch, single_layout, True, want_hash, 0, timing=True)
            assert times["2bit_lane_128_8192"][1] == 1, times
            _compare(batch, got, True, f"{kernel} hash={want_hash} family {fam}")
            n, retried = len(batch.recs), sum(retry.values())
            print(f"retries: kernel={kernel} hash={want_hash} corpus={'single' if c is single else 'doubled'} family={fam} "
                  f"records={n} retried={retried}")
            if fam == 1:
                assert retried == 0, (fam, retry)
            elif fam in (2, 3, 6):
                assert retried == (0 if pair_in_lane else n), (fam, n, retry)
            elif fam in (4, 5):
                assert retried == n, (fam, n, retry)


# ---------------------------------------------------------------- e. the doubled corpus (513 .. 8192 bases)
@pytest.mark.parametrize("aligned,no_bytes", [(True, False), (False, False), (True, True)])
def test_doubled_host_entries(ctx, doubled, aligned, no_bytes):
    got = ctx.canonicalize_batch(doubled.arena, doubled.off, want_bytes=not no_bytes, aligned=aligned)
    _compare(doubled, got, aligned, f"doubled aligned={aligned} no_bytes={no_bytes}")


def test_doubled_packed_and_uniq(ctx, doubled):
    got = ctx.canonicalize_batch_packed(doubled.arena, doubled.off, aligned=True, threads=4)
    _compare(doubled, got, True, "doubled packed")
    seqs = L.rotations_and_revcomps(doubled.seqs, np.random.default_rng(10))
    c = Corpus([L.Rec(s, -1) for s in seqs])
    wh, wfirst = oracle.uniq_consume(c.want["out"], c.off, c.want["lens"])
    ctx.uniq_reset()
    r = ctx.uniq_batch(c.arena, c.off, aligned=True)
    ctx.uniq_reset()
    assert np.array_equal(r["hash"], wh) and np.array_equal(r["first"], wfirst)
    assert (wfirst != np.arange(len(seqs))).sum() > 0.2 * len(doubled.seqs)


@pytest.mark.parametrize("want_bytes,want_hash", [(False, False), (False, True), (True, False), (True, True)])
@pytest.mark.parametrize("kernel", ["s3", "s2"])
def test_doubled_device_entry(ctx, ctx_s2, doubled, kernel, want_bytes, want_hash):
    got, _, _ = _device_run(ctx_s2 if kernel == "s2" else ctx, doubled, False, want_bytes, want_hash, 0)
    _compare(doubled, got, True, f"doubled {kernel} bytes={want_bytes} hash={want_hash}")


def test_doubled_host_entry_lane_kernel_2(ctx_s2, doubled):
    """k_canon_s2 on the doubled arena through the host entry"""
    got = ctx_s2.canonicalize_batch(doubled.arena, doubled.off, aligned=True)
    _compare(doubled, got, True, "CK_LANE_KERNEL=2 doubled")
