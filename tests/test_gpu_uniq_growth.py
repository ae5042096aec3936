"""Growth of a context's uniq first-occurrence table on the device (ck_uniq_grow / ck_uniq_table_info): first indices equal
the serial consumer's through every host entry while a table created for 16 keys grows, a growth while the other slot's
batch is in flight, one batch larger than the whole table, a stream of duplicates that does not grow the table, the
max_keys and state refusals, reset after growth, and the CLI byte for byte with a 16-key initial table.  The CPU part
checks that the header, the ctypes binding and the Rust crate agree on the two calls."""
import os
import random
import re
import shutil
import subprocess

import numpy as np
import pytest

import oracle
from oracle import cli as ocli

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu


def _records(n, seed, dup=0.3, lo=20, hi=200):
    """seeded random A/C/G/T records with rotated and reverse-complemented duplicates (a `dup` share of them)"""
    rng = np.random.default_rng(seed)
    pick = random.Random(seed)
    lens = rng.integers(lo, hi, n)
    pool = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, int(lens.sum()))].tobytes()
    seqs, pos = [], 0
    for i in range(n):
        if seqs and pick.random() < dup:
            s = pick.choice(seqs)
            r = pick.randrange(len(s))
            s = s[r:] + s[:r]
            if pick.random() < 0.5:
                s = oracle.revcomp(s)
        else:
            s = pool[pos: pos + int(lens[i])]
            pos += int(lens[i])
        seqs.append(s)
    return seqs


def _batch(seqs):
    off = np.zeros(len(seqs) + 1, dtype=np.uint64)
    np.cumsum([len(s) for s in seqs], out=off[1:])
    return np.frombuffer(b"".join(seqs), dtype=np.uint8), off


def _want(seqs):
    arena, off = _batch(seqs)
    w = oracle.canonicalize_batch(arena, off, normalize=True, threads=8)
    h, first = oracle.uniq_consume(w["out"], off, w["lens"])
    return w, h, first


def _ctx(table_capacity=16, grow=True, **kw):
    from circkit_b200.core import Context
    c = Context(**{"max_batch_bytes": 4 << 20, "max_batch_records": 4096, "table_capacity": table_capacity, **kw})
    if grow:
        c.uniq_grow()
    return c


def _code(fn, *a, **kw):
    from circkit_b200.core import CircKitError
    with pytest.raises(CircKitError) as e:
        fn(*a, **kw)
    return e.value.code


@gpu
@pytest.mark.parametrize("entry", ["submit", "packed-survivors", "fasta"])
def test_growth_from_16_keys_matches_the_serial_consumer(entry):
    from circkit_b200 import core
    seqs = _records(200_000, 1)
    want, wh, wfirst = _want(seqs)
    ctx = _ctx()
    B = 4096
    off = _batch(seqs)[1]
    try:
        cap0 = ctx.table_info()[1]
        firsts, pend = [], None

        def collect(p):
            slot, lo, hi, keep = p
            if entry == "submit":
                r = ctx.uniq_wait(slot, hi - lo, int(keep[1][-1]), want_bytes=False)
            elif entry == "packed-survivors":
                r = ctx.uniq_wait_survivors(slot, hi - lo, keep.total)
                keep_idx = np.flatnonzero(wfirst[lo:hi] == np.arange(lo, hi, dtype=np.uint64))
                assert np.array_equal(r["index"], keep_idx)
                for j, i in enumerate(r["index"].tolist()):
                    g, c0 = lo + i, int(r["offsets"][j])
                    n = int(want["lens"][g])
                    o = int(off[g])
                    assert r["bytes"][c0: c0 + n].tobytes() == want["out"][o: o + n].tobytes(), g
            else:
                r = ctx.fasta_wait(slot)
            firsts.append(r["first"])

        for b, lo in enumerate(range(0, len(seqs), B)):
            hi = min(len(seqs), lo + B)
            slot = b & 1
            if entry == "submit":
                keep = _batch(seqs[lo:hi])
                ctx.uniq_submit(slot, keep[0], keep[1], lo, normalize=True, no_bytes=True)
            elif entry == "packed-survivors":
                a, o = _batch(seqs[lo:hi])
                keep = core.pack2_host(a, o, normalize=True, threads=2)
                ctx.uniq_submit_packed(slot, keep, lo, survivors=True)
            else:
                keep = b"".join(b">r%d\n%s\n" % (lo + i, s) for i, s in enumerate(seqs[lo:hi]))
                assert ctx.fasta_submit(slot, keep, "uniq", base_index=lo) == hi - lo
            if pend is not None:
                collect(pend)
            pend = (slot, lo, hi, keep)
        collect(pend)
        assert np.array_equal(np.concatenate(firsts), wfirst)
        keys, cap, grows = ctx.table_info()
        assert keys == len(np.unique(wh))
        assert grows >= 3 and cap > 16 * cap0 and keys <= cap
    finally:
        ctx.close()


@gpu
def test_growth_while_the_other_slot_has_a_batch_in_flight():
    rng = random.Random(4)
    a = _records(3000, 2, dup=0.1)
    b = []
    for i in range(6000):                                      # half of B repeats A's records, rotated / reverse-complemented
        if i % 2:
            s = rng.choice(a)
            r = rng.randrange(len(s))
            s = s[r:] + s[:r]
            b.append(oracle.revcomp(s) if rng.random() < 0.5 else s)
        else:
            b.append(bytes(rng.choice(b"ACGT") for _ in range(rng.randint(20, 120))))
    a[::7] = [oracle.revcomp(s) for s in b[::2][: len(a[::7])]]   # and some of B's new records appear first in A
    seqs = a + b
    _, _, wfirst = _want(seqs)
    ctx = _ctx(table_capacity=4000, max_batch_records=8192)
    try:
        pa, pb = _batch(a), _batch(b)
        ctx.uniq_submit(0, pa[0], pa[1], 0, normalize=True, no_bytes=True)
        ctx.uniq_submit(1, pb[0], pb[1], len(a), normalize=True, no_bytes=True)   # A unwaited: B's submit grows the table
        ra = ctx.uniq_wait(0, len(a), int(pa[1][-1]), want_bytes=False)
        rb = ctx.uniq_wait(1, len(b), int(pb[1][-1]), want_bytes=False)
        assert np.array_equal(ra["first"], wfirst[: len(a)])
        assert np.array_equal(rb["first"], wfirst[len(a):])
        assert ctx.table_info()[2] == 1
    finally:
        ctx.close()


@gpu
def test_one_batch_larger_than_the_whole_table():
    seqs = _records(100_000, 3, dup=0.0, lo=40, hi=80)
    _, wh, wfirst = _want(seqs)
    assert len(np.unique(wh)) == len(seqs)
    ctx = _ctx(max_batch_records=1 << 17, max_batch_bytes=16 << 20)
    try:
        arena, off = _batch(seqs)
        r = ctx.uniq_batch(arena, off, 0, normalize=True, want_bytes=False)
        assert np.array_equal(r["first"], wfirst)
        keys, cap, grows = ctx.table_info()
        assert keys == len(seqs) and cap >= len(seqs) and grows == 1
    finally:
        ctx.close()


@gpu
def test_a_stream_of_duplicates_keeps_the_size_the_first_batch_needed():
    seqs = _records(1000, 5)
    _, wh, wfirst = _want(seqs)
    arena, off = _batch(seqs)
    ctx = _ctx()
    try:
        ctx.uniq_submit(0, arena, off, 0, normalize=True, no_bytes=True)
        assert np.array_equal(ctx.uniq_wait(0, 1000, int(off[-1]), want_bytes=False)["first"], wfirst)
        first_info = ctx.table_info()
        assert first_info[0] == len(np.unique(wh)) and first_info[2] == 1
        pend = None
        for k in range(1, 50):
            ctx.uniq_submit(k & 1, arena, off, 1000 * k, normalize=True, no_bytes=True)
            if pend is not None:
                assert np.array_equal(ctx.uniq_wait(pend, 1000, int(off[-1]), want_bytes=False)["first"], wfirst)
            pend = k & 1
        assert np.array_equal(ctx.uniq_wait(pend, 1000, int(off[-1]), want_bytes=False)["first"], wfirst)
        assert ctx.table_info() == first_info
    finally:
        ctx.close()


@gpu
def test_max_keys_refuses_the_batch_and_keeps_the_table():
    from circkit_b200 import _native as N
    seqs = _records(5000, 6, dup=0.0)
    _, wh, wfirst = _want(seqs)
    assert len(np.unique(wh)) == 5000
    ctx = _ctx(grow=False)
    try:
        ctx.uniq_grow(max_keys=3000)
        a, o = _batch(seqs[:2000])
        r = ctx.uniq_batch(a, o, 0, normalize=True, want_bytes=False)
        assert np.array_equal(r["first"], wfirst[:2000])
        info = ctx.table_info()
        b, p = _batch(seqs[2000:])
        assert _code(ctx.uniq_submit, 0, b, p, 2000, normalize=True, no_bytes=True) == N.CK_ERR_TABLE_FULL
        assert "max_keys" in ctx._lib.ck_last_error(ctx.handle).decode()
        assert ctx.table_info() == info
        r = ctx.uniq_batch(a[: int(o[1000])], o[:1001], 10_000, normalize=True, want_bytes=False)   # the slot is usable
        assert np.array_equal(r["first"], wfirst[:1000])
    finally:
        ctx.close()


@gpu
def test_a_fixed_table_still_fills_up_at_the_wait():
    from circkit_b200 import _native as N
    seqs = _records(2000, 7, dup=0.0)
    a, o = _batch(seqs)
    ctx = _ctx(grow=False)
    try:
        assert ctx.table_info()[1] < 2000
        ctx.uniq_submit(0, a, o, 0, normalize=True, no_bytes=True)
        assert _code(ctx.uniq_wait, 0, 2000, int(o[-1]), want_bytes=False) == N.CK_ERR_TABLE_FULL
        assert ctx.table_info()[2] == 0
    finally:
        ctx.close()


@gpu
def test_state_refusals():
    from circkit_b200 import _native as N
    none = _ctx(table_capacity=0, grow=False)
    try:
        assert _code(none.uniq_grow) == N.CK_ERR_STATE
    finally:
        none.close()
    peer = _ctx(grow=False)
    try:
        peer.peer_attach([peer.peer_export(1, 0, 16)])                 # a peer group of one
        assert _code(peer.uniq_grow) == N.CK_ERR_STATE
    finally:
        peer.close()
    grown = _ctx()
    try:
        assert _code(grown.peer_export, 1, 0, 16) == N.CK_ERR_STATE
    finally:
        grown.close()


@gpu
def test_reset_after_growth_keeps_the_size():
    seqs = _records(20_000, 8)
    _, wh, wfirst = _want(seqs)
    a, o = _batch(seqs)
    ctx = _ctx(max_batch_records=1 << 15)
    try:
        ctx.uniq_batch(a, o, 0, normalize=True, want_bytes=False)
        keys, cap, grows = ctx.table_info()
        assert keys == len(np.unique(wh)) and grows >= 1
        ctx.uniq_reset()
        assert ctx.table_info() == (0, cap, grows)
        r = ctx.uniq_batch(a[: int(o[5000])], o[:5001], 0, normalize=True, want_bytes=False)
        _, _, w5 = _want(seqs[:5000])
        assert np.array_equal(r["first"], w5)
        assert ctx.table_info()[0] == len(np.unique(wh[:5000])) and ctx.table_info()[1] == cap
    finally:
        ctx.close()


def _synthetic(n, seed):
    """wrapped lines, CRLF, lower case, RNA, rotated / reverse-complemented duplicates"""
    rng = random.Random(seed)
    recs, out = [], []
    for i in range(n):
        if recs and rng.random() < 0.3:
            s = rng.choice(recs)
            r = rng.randrange(len(s))
            s = s[r:] + s[:r]
            if rng.random() < 0.5:
                s = oracle.revcomp(s)
        else:
            s = bytes(rng.choice(b"ACGT") for _ in range(rng.randint(1, 300)))
            recs.append(s)
        if rng.random() < 0.1:
            s = s.lower()
        if rng.random() < 0.05:
            s = s.replace(b"T", b"U")
        eol = b"\r\n" if rng.random() < 0.1 else b"\n"
        w = rng.choice([0, 60, 70])
        body = eol.join(s[k:k + w] for k in range(0, len(s), w)) if w else s
        out.append(b">r%d some description" % i + eol + body + eol)
    return b"".join(out)


@gpu
@pytest.mark.parametrize("canonical", [False, True], ids=["raw-body", "canonical-body"])
def test_cli_from_a_16_key_table(tmp_path, monkeypatch, canonical):
    from circkit_b200 import cli
    monkeypatch.setattr(cli, "UNIQ_TABLE_KEYS", 16)
    text = _synthetic(6000, 9 + canonical)
    want, want_table = ocli.cli_uniq(text, canonical, "csv")
    src, out, tab = tmp_path / "in.fa", tmp_path / "out.fa", tmp_path / "t.csv"
    src.write_bytes(text)
    argv = ["uniq", str(src), "-o", str(out), "--table", str(tab)] + (["-c"] if canonical else [])
    assert cli.main(argv) == 0
    assert out.read_bytes() == want and tab.read_bytes() == want_table
    cuts = [0] + [m.start() + 1 for m in re.finditer(rb"\n>", text)][::50] + [len(text)]   # pieces of 50 records
    got, table = [], []
    cli.run_uniq([text[lo:hi] for lo, hi in zip(cuts, cuts[1:]) if hi > lo], got.append, canonical, table.append, "csv")
    assert b"".join(got) == want and b"".join(table) == want_table


def test_header_binding_and_crate_agree_on_the_growth_calls(tmp_path):
    from circkit_b200 import _native
    hdr = open(os.path.join(ROOT, "include", "circkit_b200.h")).read()
    assert re.search(r"int ck_uniq_grow\(ck_ctx \*ctx, uint64_t max_keys\);", hdr)
    assert re.search(r"int ck_uniq_table_info\(ck_ctx \*ctx, uint64_t \*out_keys, uint64_t \*out_capacity_keys, "
                     r"uint64_t \*out_grows\);", hdr)
    if shutil.which("gcc"):
        src = tmp_path / "probe.c"
        src.write_text('#include "circkit_b200.h"\nint main(void) {\n'
                       '    int (*grow)(ck_ctx *, uint64_t) = 0;\n'
                       '    int (*info)(ck_ctx *, uint64_t *, uint64_t *, uint64_t *) = 0;\n'
                       '    (void)sizeof(grow = ck_uniq_grow); (void)sizeof(info = ck_uniq_table_info);\n'
                       '    return 0;\n}\n')
        subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-Wno-unused-but-set-variable", "-I",
                        os.path.join(ROOT, "include"), "-o", str(tmp_path / "probe"), str(src)], check=True)
    assert len(_native.SIGNATURES["ck_uniq_grow"][1]) == 2 and len(_native.SIGNATURES["ck_uniq_table_info"][1]) == 4
    rs = open(os.path.join(ROOT, "circkit-cuda", "src", "lib.rs")).read()
    assert re.search(r"pub fn ck_uniq_grow\(ctx: \*mut CkCtx, max_keys: u64\) -> c_int;", rs)
    assert re.search(r"pub fn ck_uniq_table_info\(ctx: \*mut CkCtx, out_keys: \*mut u64, out_capacity_keys: \*mut u64, "
                     r"out_grows: \*mut u64\) -> c_int;", rs)
    assert re.search(r"ctx\.uniq_grow\(None\)\?;", rs)                # Pump turns growth on
