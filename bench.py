#!/usr/bin/env python
"""bench.py -- canonicalize+uniq throughput of the B200 hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torch.distributed.run)
  python bench.py --impl reference ...                     (CPU arm: the oracle port of circKit's path)
  python bench.py ... --dump-outputs DIR                   (also write the last timed step's results as DIR/*.npy)

A step = one pass of the hot path over one batch of synthetic records:
  config 2 of BASELINE.json (default): `circkit uniq` on 10 M circRNA-length records (log-uniform
  0.2-5 kb, 30 % duplicates as random rotations / reverse complements), per GPU (weak scaling);
  the batch is resident in HBM as a packed 2-bit arena when the timed region starts (`value`);
  `e2e` runs the same records through the host-buffer C ABI (ck_uniq_submit / ck_uniq_wait) from pinned
  host memory, copies included.
Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (records per GPU, length law, lo, hi, dup permille, adversarial permille, uniq?, class mask)
    "c1": dict(records=1_000_000, kind=0, lo=250, hi=400, dup=0, adv=0, uniq=False,
               desc="config 1: canonicalize, 1M viroid-length (250-400 nt) records"),
    "c2": dict(records=10_000_000, kind=1, lo=200, hi=5000, dup=300, adv=0, uniq=True,
               desc="config 2: uniq, 10M circRNA-length (0.2-5 kb log-uniform) records, 30% rotated/revcomp duplicates"),
    "c3": dict(records=5_000_000, kind=0, lo=250, hi=400, dup=0, adv=0, uniq=False, raw=True,
               desc="config 3: canonicalize, 5M mixed IUPAC/N records (byte-level lanes, CLI semantics: normalise on device)"),
    "c4": dict(records=200_000, kind=1, lo=5000, hi=200_000, dup=0, adv=10, uniq=False,
               desc="config 4: canonicalize, 200k plasmid/mtDNA-length (5-200 kb) records, 1% adversarial repeats"),
    "c5": dict(records=12_500_000, kind=0, lo=250, hi=400, dup=300, adv=0, uniq=True,
               desc="config 5: uniq, 100M viroid-length records over 8 GPUs (12.5M per GPU), 30% duplicates"),
}
SEEDS = {"c1": 1, "c2": 2, "c3": 3, "c4": 4, "c5": 5}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS) + ["mono"])
    ap.add_argument("--records", type=int, default=0, help="override records per GPU (smaller = NOT the named config)")
    ap.add_argument("--e2e-ascii-every", type=int, default=None,
                    help="e2e: every k-th batch goes to the device as ASCII (ck_*_submit: the DMA engine moves it while the host threads "
                         "pack the other batches, ck_pack2_host + ck_*_submit_packed) -- host packing (~70 GB/s of ASCII on 16 threads) and "
                         "PCIe (~55 GB/s) work side by side instead of one after the other; 0 = every batch packed on the host.  Default 3; "
                         "config 3 (IUPAC records: nothing to gain from 2-bit packing on the host): 1 = every batch as ASCII")
    ap.add_argument("--no-config5", action="store_true", help="default workload only: skip the 100 M-record config-5 sub-record")
    ap.add_argument("--c5-records", type=int, default=100_000_000, help="records of the config-5 sub-record, split over the GPUs")
    ap.add_argument("--overlap", dest="overlap", action="store_true", default=None,
                    help="uniq: run the table / exchange stage of a step on a second stream with double-buffered outputs, so that "
                         "it overlaps the canonicalisation of the next step.  Default: on with more than one GPU (round 2, 2 GPUs: "
                         "config 2 +3.4 %%, config 5 +6-7 %%), off on one GPU (+1 %%, and the kernel timings of the roofline then "
                         "include the table's traffic)")
    ap.add_argument("--no-overlap", dest="overlap", action="store_false")
    ap.add_argument("--exchange", default="peer", choices=["peer", "symm", "padded", "exact"],
                    help="multi-GPU uniq, how (hash, index) pairs reach their owner: peer = stored straight into the owner's buffer by "
                         "the partition kernel over NVLink (fixed-capacity buckets, device-side barriers, no collective); padded = "
                         "the same buckets through one equal-split NCCL all-to-all each way; exact = per-owner counts exchanged first "
                         "(two host synchronisations per step)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU work per cpu_baseline measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs), so that "
                         "two builds can be compared output for output on the same inputs; B200 arm only")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs: the reference arm times a host-side sample, not the B200 path")
    return args


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe).  nvidia-smi needs
    ~100 ms to come up and the timed region of the short configurations lasts a few ms, so the sampler starts early
    (20 ms period) and `stop(t0, t1)` keeps the samples that arrived between the start of the warm-up and the end
    of the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def stop(self, t0: float = 0.0, t1: float = float("inf")):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        window = [ln for ts, ln in self.lines if t0 <= ts <= t1 + 0.03]
        sm, mx, reasons = [], [], set()
        for ln in window:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        # median over the samples taken under load (upper half of the clock samples in the window)
        load = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
def cpu_arm(w, seed, cpu_seconds, steps, warmup, uniq):
    """circKit's CPU path (oracle port, O(1)-indexed Duval) on a bounded sample of the workload.

    Worker stage (normalise + canonicalize, src/uniq.rs:33-41) on all host cores; consumer stage
    (xxh3 + first-occurrence map, src/uniq.rs:42-78) single-threaded as in the reference.  The two
    overlap in the reference (parallel_fasta pipelines them), so a step's time is max(worker, consumer)."""
    import numpy as np
    import oracle
    from oracle import synth
    cores = oracle.max_threads()
    pilot_n = 2000
    a, o = synth.make_records(pilot_n, w["kind"], w["lo"], w["hi"], w["dup"], seed)
    t = time.perf_counter()
    oracle.canonicalize_batch(a, o, normalize=True, threads=cores, want_start=False, want_hash=False)
    rate = pilot_n / max(time.perf_counter() - t, 1e-6)
    per_step = max(cpu_seconds / max(steps + warmup, 1), 0.5)
    n = int(min(max(rate * per_step, 2000), 2_000_000))
    a, o = synth.make_records(n, w["kind"], w["lo"], w["hi"], w["dup"], seed)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        r = oracle.canonicalize_batch(a, o, normalize=True, threads=cores, want_start=False, want_hash=False)
        t1 = time.perf_counter()
        if uniq:
            oracle.uniq_consume(r["out"], o, r["lens"])
        t2 = time.perf_counter()
        if it >= warmup:
            times.append(max(t1 - t0, t2 - t1))
    sec = sum(times) / len(times)
    bases = int(o[-1])
    return dict(records_per_s=n / sec, gbases_per_s=bases / sec / 1e9, cores=cores, sample_records=n,
                sample_bases=bases, ms_per_step=sec * 1e3)


def cpu_faithful_footnote(w, seed):
    """The reference AS WRITTEN indexes with s.chars().nth(i) (O(i) per access, lib/src/canonicalize.rs:18-25):
    time that on a tiny sample and report records/s per core (extrapolated, labelled as such)."""
    import oracle
    from oracle import synth
    n = 40 if w["hi"] <= 5000 else 2
    a, o = synth.make_records(n, w["kind"], w["lo"], min(w["hi"], 20000), 0, seed)
    t = time.perf_counter()
    oracle.canonicalize_batch(a, o, normalize=True, threads=1, want_start=False, want_hash=False, faithful_cost=True)
    dt = time.perf_counter() - t
    return {"records_per_s_per_core": n / dt, "sample_records": n, "note": "extrapolated; O(n^2) chars().nth emulation"}


# ------------------------------------------------------------------------------------------------
DUMP_RECORDS = 1 << 18      # --dump-outputs: per-record results of at most this many records
DUMP_BASES = 1 << 21        # --dump-outputs: canonical bytes of at most this many bases


def dump_outputs(dirname, prefix, n, per_record, canon=None):
    """--dump-outputs: the results of the last timed step, for all n records or, above DUMP_RECORDS, for a sample drawn with
    a fixed seed, as DIR/<prefix><name>.npy:
      index            the sampled record indices (float64)
      <name>           per_record[name][index] for each device array of n per-record results (float64: exact below 2^53);
                       the 64-bit hash as hash_hi and hash_lo, its two 32-bit halves
      canonical_bytes  (canon given) the canonical bytes of the first sampled records that fit DUMP_BASES, concatenated
                       (float32); per_record["length"] splits them
    canon = (out, offsets): the aligned output arena, record i at 32 * ((offsets[i] >> 5) + i)."""
    import numpy as np
    import torch
    idx = np.arange(n) if n <= DUMP_RECORDS else np.sort(np.random.default_rng(0).choice(n, DUMP_RECORDS, replace=False))
    res = {"index": idx.astype(np.float64)}
    didx = torch.from_numpy(idx).to(next(iter(per_record.values())).device)
    for name, t in per_record.items():
        v = t[:n][didx].cpu().numpy()
        if name == "hash":
            u = v.view(np.uint64)
            res["hash_hi"], res["hash_lo"] = (u >> np.uint64(32)).astype(np.float64), (u & np.uint64(0xFFFFFFFF)).astype(np.float64)
        else:
            res[name] = v.astype(np.float64)
    if canon is not None:
        out, offsets = canon
        lens = per_record["length"][:n][didx].long()
        ends = torch.cumsum(lens, 0)
        m = int((ends <= DUMP_BASES).sum().item())
        starts = 32 * ((offsets[didx[:m]] >> 5) + didx[:m])
        total = int(ends[m - 1].item()) if m else 0
        pos = torch.repeat_interleave(starts - (ends[:m] - lens[:m]), lens[:m]) + torch.arange(total, device=out.device)
        res["canonical_bytes"] = out[pos].cpu().numpy().astype(np.float32)
    os.makedirs(dirname, exist_ok=True)
    for name, a in res.items():
        np.save(os.path.join(dirname, prefix + name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
def bench_monomerize(args):
    """`--workload mono`: `monomerize` (SURVEY 8f row 4) on one GPU.  1 M concatemers (2.3 copies of a 250-400 nt unit, 1 %
    substitutions; `--records` overrides), seed 10, min identity 0.95 (the reference CLI's default seed, its tests' identity).
    value: resident bytes -> end indices (k_monomerize); e2e: pinned host bytes + offsets -> H2D -> kernel -> D2H of the end
    indices; cpu_baseline: the compiled oracle port (oracle/ck_oracle.c: ck_o_monomerize_batch) on all host threads over a
    bounded sample, whose answers are also compared with the GPU's."""
    import numpy as np
    import torch
    import circkit_b200
    from circkit_b200.monomerize import Monomerizer
    n = args.records or 1_000_000
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    sampler = ClockSampler(0)
    sampler.start()
    rng = np.random.default_rng(1)
    unit_len = rng.integers(250, 401, n)
    total_len = (unit_len * 2.3).astype(np.int64)
    off = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(total_len, out=off[1:])
    T = int(off[-1])
    offsets = torch.from_numpy(off).to(dev)
    rec = torch.repeat_interleave(torch.arange(n, device=dev), torch.from_numpy(total_len).to(dev))
    pos = torch.arange(T, device=dev) - offsets[rec]
    h = (rec * 1000003 + (pos % torch.from_numpy(unit_len).to(dev)[rec])) * 2654435761 % 4294967296
    letters = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device=dev)
    raw = letters[((h >> 13) ^ (h >> 7)) & 3]
    g = torch.Generator(device=dev).manual_seed(7)
    mut = torch.rand(T, device=dev, generator=g) < 0.01
    raw[mut] = letters[torch.randint(0, 4, (int(mut.sum()),), device=dev, generator=g)]
    del rec, pos, h, mut
    ctx = circkit_b200.Context(max_batch_bytes=0, max_batch_records=0)
    m = Monomerizer(10, overlap_min_identity=0.95, ctx=ctx)
    t0 = time.time()
    for _ in range(args.warmup):
        out = m.end_indices_device(raw, offsets, n)
    torch.cuda.synchronize()
    launches0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = m.end_indices_device(raw, offsets, n)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    launches = ctx.launch_count() - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, "", n, {"end_index": out})       # -1: no monomer found
    # end to end: host buffers in, end indices out
    h_raw = raw.cpu().pin_memory(); h_off = offsets.cpu().pin_memory()
    h_out = torch.empty(n, dtype=torch.int32).pin_memory()
    d_raw, d_off = torch.empty_like(raw), torch.empty_like(offsets)
    e2e_steps = max(1, min(args.steps, 3))
    torch.cuda.synchronize()
    te = time.perf_counter()
    for _ in range(e2e_steps):
        d_raw.copy_(h_raw, non_blocking=True); d_off.copy_(h_off, non_blocking=True)
        h_out.copy_(m.end_indices_device(d_raw, d_off, n), non_blocking=True)
        torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - te) / e2e_steps
    clocks = sampler.stop(t0, time.time())
    peak, src = 6551.7, "fallback"
    pp = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pp):
        peak, src = float(json.load(open(pp)).get("hbm_gbs", peak)), "measured (MEASURED_PEAKS.json hbm_gbs)"
    alg = T + 12 * n                                        # record bytes read once + offsets + the end index
    cpu = None
    if not args.no_cpu:
        from oracle.monomerize import c_end_indices_batch
        k = min(n, 200_000)
        a_np, o_np = h_raw[: int(off[k])].numpy(), off[: k + 1].astype(np.uint64)
        threads = os.cpu_count() or 1
        c_end_indices_batch(a_np[: int(off[1000])], o_np[:1001], 10, None, 0.95, False, threads)
        tc = time.perf_counter()
        want = c_end_indices_batch(a_np, o_np, 10, None, 0.95, False, threads)
        tc = time.perf_counter() - tc
        same = bool((want == out[:k].cpu().numpy().astype(np.uint32)).all())
        cpu = {"value": k / tc, "unit": "records/s", "cores": threads, "kind": "port",
               "sample": "%d records (%.0f Mbases) of the workload, compiled oracle port (memmem seed search + byte Hamming), "
                         "all host threads; its end indices equal the GPU's: %s" % (k, off[k] / 1e6, same)}
        if not same:
            raise RuntimeError("GPU and CPU port disagree on the bench sample")
    print(json.dumps({
        "metric": "monomerize records/sec", "value": n / (ms / 1e3), "unit": "records/s", "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic", "config": {"workload": "monomerize: %d concatemers (2.3 copies of a 250-400 nt unit, 1%% substitutions), "
                                                    "seed 10, min identity 0.95" % n, "records_per_gpu": n,
                                        "l2_policy": "inputs larger than L2 (%.2f GB of record bytes per step)" % (T / 1e9)},
        "gbases_per_s": T / ms / 1e6, "clocks": clocks,
        "e2e": {"value": n / e2e_s, "unit": "records/s", "h2d_bytes_per_step": T + 8 * (n + 1), "d2h_bytes_per_step": 4 * n,
                "steps": e2e_steps, "api": "ck_dev_monomerize after H2D of pinned record bytes + offsets"},
        "gpu_launches": launches,
        "roofline": {"bound": "hbm", "kernel": "k_monomerize (warp per record)", "achieved": alg / ms / 1e6, "peak": peak,
                     "unit": "GB/s", "frac": alg / ms / 1e6 / peak, "traffic": None, "peak_source": src,
                     "algorithmic_bytes_per_launch": alg, "kernel_ms_per_launch": ms, "launches_per_step": 1.0},
        "cpu_baseline": cpu, "monomerized_records": int((out != -1).sum())}))
    ctx.close()


def bench_monomerize_reference(args):
    """`--workload mono --impl reference`: the compiled oracle port of lib/src/monomerize.rs:50-141 on all host threads; each
    step is a bounded sample (200 k records) of the same concatemer workload, generated on the host with the same law."""
    import numpy as np
    from oracle.monomerize import c_end_indices_batch
    k = min(args.records or 1_000_000, 200_000)
    rng = np.random.default_rng(1)
    unit_len = rng.integers(250, 401, k)
    total_len = (unit_len * 2.3).astype(np.int64)
    off = np.zeros(k + 1, dtype=np.uint64)
    np.cumsum(total_len, out=off[1:])
    T = int(off[-1])
    rec = np.repeat(np.arange(k, dtype=np.int64), total_len)
    pos = np.arange(T, dtype=np.int64) - off[:-1].astype(np.int64)[rec]
    h = (rec * 1000003 + (pos % unit_len[rec])) * 2654435761 % 4294967296
    arena = np.frombuffer(b"ACGT", dtype=np.uint8)[((h >> 13) ^ (h >> 7)) & 3].copy()
    mut = rng.random(T) < 0.01
    arena[mut] = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, int(mut.sum()))]
    threads = os.cpu_count() or 1
    for _ in range(max(args.warmup, 1)):
        out = c_end_indices_batch(arena, off, 10, None, 0.95, False, threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = c_end_indices_batch(arena, off, 10, None, 0.95, False, threads)
    dt = (time.perf_counter() - t0) / args.steps
    v = k / dt
    sample = "%d records (%.0f Mbases) per step, compiled oracle port (memmem seed search + byte Hamming), %d host threads" % (k, T / 1e6, threads)
    print(json.dumps({
        "impl": "reference", "metric": "monomerize records/sec", "value": v, "unit": "records/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "monomerize: concatemers (2.3 copies of a 250-400 nt unit, 1% substitutions), seed 10, min identity 0.95",
                   "records_per_step": k},
        "cpu_baseline": {"value": v, "unit": "records/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "records/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "monomerized_records": int((out != 0xffffffff).sum())}))


def e2e_leg(args, ctx, D, torch, dist, dev, rank, world, w, wname, R, resident_first, sync_all, steps):
    """The same metric end to end through the host-buffer C ABI, copies and host packing inside the timed region:
    pinned ASCII record bytes -> ck_pack2_host (normalise + classify + 2-bit pack, all host threads of this rank) ->
    ck_uniq_submit_packed / ck_canon_submit_packed (H2D of a quarter of the bytes, kernels) -> ck_*_wait (D2H of the results).
    Batches alternate between the two slots, so packing, copies and kernels of consecutive batches overlap.
    world > 1: GLOBAL uniq through the library's peer group (ck_peer_export / ck_peer_attach): batch k of the input goes to
    rank k % world in round k // world, every round is one collective exchange, first indices are exact at every wait."""
    import ctypes as C
    import numpy as np
    from circkit_b200 import _native as N
    lib = ctx._lib
    seed = SEEDS[wname]
    uniq = w["uniq"]
    raw = bool(w.get("raw"))
    RB = 1 << 17 if w["hi"] > 1000 else 1 << 19          # records per batch (<= max_batch_records, bytes <= max_batch_bytes)
    if w["hi"] > 50_000:
        RB = 1 << 11
    total_records = R * world
    n_batches = (total_records + RB - 1) // RB
    mine = list(range(rank, n_batches, world))             # this rank's batches of the global input
    rounds = (n_batches + world - 1) // world
    # every rank pins its own input: bound it to ~4 GiB of record bytes per rank when there are several (the first rounds of
    # the input -- the same steady-state batches, fewer of them; first indices of a prefix are those of the whole run)
    mean_len = (w["lo"] + w["hi"]) / 2 if w["kind"] == 0 else (w["hi"] - w["lo"]) / np.log(w["hi"] / w["lo"])
    if world > 1:
        rounds = max(1, min(rounds, int((4 << 30) / (RB * mean_len))))
    mine = [k for k in mine if k // world < rounds]
    if world > 1 and uniq and not getattr(ctx, "_peer_attached", False):
        handles = [None] * world
        dist.all_gather_object(handles, ctx.peer_export(world, rank, ctx.max_batch_records))
        ctx.peer_attach(handles)
        ctx._peer_attached = True
    threads = max(1, (os.cpu_count() or 1) // world)
    # ---- this rank's batches as pinned ASCII + offsets
    batches = []
    for k in mine:
        lo_i = k * RB
        n_k = min(RB, total_records - lo_i)
        if raw:
            from circkit_b200 import synth_host
            a_np, o_np = synth_host.make_iupac_records(n_k, w["lo"], w["hi"], seed + 1000 + k)
            tot = int(o_np[-1])
            hp = lib.ck_alloc_pinned(ctx.handle, tot + 64)
            hb = np.ctypeslib.as_array(C.cast(hp, C.POINTER(C.c_uint8)), shape=(tot + 64,))
            hb[:tot] = a_np
            off = o_np.astype(np.uint64)
        else:
            b = D.synth_batch(ctx, seed=seed, first_index=lo_i, n_records=n_k, kind=w["kind"], lo=w["lo"], hi=w["hi"],
                              dup_permille=w["dup"], adversarial_permille=w["adv"], device=dev)
            asc = D.unpack_ascii(ctx, b)
            tot = b.total
            hp = lib.ck_alloc_pinned(ctx.handle, tot + 64)
            hb = np.ctypeslib.as_array(C.cast(hp, C.POINTER(C.c_uint8)), shape=(tot + 64,))
            torch.from_numpy(hb)[:tot].copy_(asc)
            off = b.offsets.cpu().numpy().astype(np.uint64)
            del b, asc
        op = lib.ck_alloc_pinned(ctx.handle, off.nbytes)
        oarr = np.ctypeslib.as_array(C.cast(op, C.POINTER(C.c_uint64)), shape=(len(off),))
        oarr[:] = off
        batches.append(dict(k=k, lo=lo_i, n=n_k, total=tot, bytes_p=hp, off=oarr, off_p=op))
    torch.cuda.synchronize()
    max_total = max([b["total"] for b in batches] + [1])
    max_n = max([b["n"] for b in batches] + [1])
    # ---- three packed staging sets (pinned): dense words, lens, lanes, byte-lane bytes + offsets
    sets = []
    for _ in range(3):
        words = int(lib.ck_pack2_words(max_total, max_n))
        s = dict(dense=lib.ck_alloc_pinned(ctx.handle, 8 * words), lens=lib.ck_alloc_pinned(ctx.handle, 4 * max_n + 16),
                 lane=lib.ck_alloc_pinned(ctx.handle, max_n + 16), lane_off=lib.ck_alloc_pinned(ctx.handle, 8 * (max_n + 1)),
                 lane_bytes=lib.ck_alloc_pinned(ctx.handle, (max_total if raw else (1 << 20)) + 64),
                 lane_cap=(max_total if raw else (1 << 20)), total=C.c_uint64(0), st=None)
        sets.append(s)
    n_mine = sum(b["n"] for b in batches)
    out_first_p = lib.ck_alloc_pinned(ctx.handle, 8 * (n_mine + 1))
    out_hash_p = lib.ck_alloc_pinned(ctx.handle, 8 * (n_mine + 1))
    out_len_p = lib.ck_alloc_pinned(ctx.handle, 4 * (n_mine + 1))
    out_start_p = lib.ck_alloc_pinned(ctx.handle, 4 * (n_mine + 1))
    out_strand_p = lib.ck_alloc_pinned(ctx.handle, (n_mine + 1))
    pos = [0]
    for b in batches:
        pos.append(pos[-1] + b["n"])
    # CK_F_NO_BYTES: `circkit uniq` without -c echoes the input bytes; result = first_index per record (config 3: + CK_F_NORMALIZE)
    sub_flags = 2
    pack_flags = 1 if raw else 0
    stats = dict(pack_s=0.0, h2d=0)

    sched = dict(every=max(0, args.e2e_ascii_every) if args.e2e_ascii_every is not None else (1 if raw else 3))

    def is_ascii(i):
        every = sched["every"]
        return every > 0 and i % every == every - 1

    def pack(i):
        if is_ascii(i):
            return
        b, s = batches[i], sets[i % 3]
        t0 = time.perf_counter()
        rc = lib.ck_pack2_host(b["bytes_p"], b["off_p"], b["n"], pack_flags, threads, s["dense"], s["lens"], s["lane"], s["lane_bytes"],
                               s["lane_cap"], s["lane_off"], C.byref(s["total"]))
        stats["pack_s"] += time.perf_counter() - t0
        if rc != 0:
            raise RuntimeError("ck_pack2_host failed: %d" % rc)
        lt = int(s["total"].value)
        s["st"] = N.CkPackedBatch(s["dense"], b["off_p"], s["lens"], s["lane"], s["lane_bytes"] if lt else None,
                                  s["lane_off"] if lt else None, lt, b["n"])
        stats["h2d"] += 8 * int(lib.ck_pack2_words(b["total"], b["n"])) + 8 * (b["n"] + 1) + 5 * b["n"] + (lt + 8 * (b["n"] + 1) if lt else 0)

    empty = N.CkPackedBatch(None, None, None, None, None, None, 0, 0)

    def submit(j):                                        # round j: this rank's batch, or an empty one (the rounds are collective)
        i = j if world == 1 else j
        if i < len(batches) and is_ascii(i):
            b = batches[i]
            stats["h2d"] += b["total"] + 8 * (b["n"] + 1)
            if uniq:
                ctx._check(lib.ck_uniq_submit(ctx.handle, j & 1, b["bytes_p"], b["off_p"], b["n"], sub_flags | pack_flags, b["lo"]))
            else:
                ctx._check(lib.ck_canon_submit(ctx.handle, j & 1, b["bytes_p"], b["off_p"], b["n"], sub_flags | pack_flags))
        elif i < len(batches):
            b, s = batches[i], sets[i % 3]
            if uniq:
                ctx._check(lib.ck_uniq_submit_packed(ctx.handle, j & 1, C.byref(s["st"]), sub_flags, b["lo"]))
            else:
                ctx._check(lib.ck_canon_submit_packed(ctx.handle, j & 1, C.byref(s["st"]), sub_flags))
        else:
            ctx._check(lib.ck_uniq_submit_packed(ctx.handle, j & 1, C.byref(empty), sub_flags, 0))

    def wait(j):
        if j < len(batches):
            c0 = pos[j]
            if uniq:
                ctx._check(lib.ck_uniq_wait(ctx.handle, j & 1, None, out_len_p + 4 * c0, out_hash_p + 8 * c0, out_first_p + 8 * c0))
            else:
                ctx._check(lib.ck_canon_wait(ctx.handle, j & 1, None, out_len_p + 4 * c0, out_start_p + 4 * c0, out_strand_p + c0, None))
        else:
            ctx._check(lib.ck_uniq_wait(ctx.handle, j & 1, None, None, None, None))

    n_rounds = rounds if (world > 1 and uniq) else len(batches)

    def e2e_step():
        if uniq:
            ctx.uniq_reset()
            if world > 1:
                dist.barrier()
        stats["pack_s"], stats["h2d"] = 0.0, 0
        if batches:
            pack(0)
        for j in range(n_rounds):
            submit(j)
            if j + 1 < len(batches):
                pack(j + 1)                                # the host packs the next batch while the device works on this one
            if j >= 1:
                wait(j - 1)
        if n_rounds:
            wait(n_rounds - 1)

    e2e_step()                         # warm-up
    sync_all()
    probe = None
    if args.e2e_ascii_every is None and not raw:
        # the share of batches that cross PCIe as ASCII is a property of the host (packer threads vs. DMA engine vs. memory
        # bandwidth): one untimed step per candidate, the same choice on every rank
        probe = {}
        for cand in (3, 2, 1, 4, 6, 0):
            sched["every"] = cand
            e2e_step()
            sync_all()
            tq = time.perf_counter()
            e2e_step()
            torch.cuda.synchronize()
            dq = time.perf_counter() - tq
            if world > 1:
                t = torch.tensor([dq], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dq = float(t.item())
            probe[cand] = dq
            sync_all()
        sched["every"] = min(probe, key=probe.get)
        e2e_step()
        sync_all()
    every = sched["every"]
    t0 = time.perf_counter()
    e2e_steps = max(1, min(steps, 3))
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([dt], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    # ---- the same path with the packing done beforehand (what a host whose reader threads pack while they parse FASTA --
    #      the north star's host side -- hands over): the first batches of the input, each in its own packed staging set
    prepacked = None
    npre = min(len(batches), 12)
    if world > 1:                                          # the rounds are collective: every rank takes the same number
        t = torch.tensor([npre], dtype=torch.int64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        npre = int(t.item())
    if npre:
        pre_sets = []
        for i in range(npre):
            b = batches[i]
            words = int(lib.ck_pack2_words(b["total"], b["n"]))
            ps = dict(dense=lib.ck_alloc_pinned(ctx.handle, 8 * words), lens=lib.ck_alloc_pinned(ctx.handle, 4 * b["n"] + 16),
                      lane=lib.ck_alloc_pinned(ctx.handle, b["n"] + 16), lane_off=lib.ck_alloc_pinned(ctx.handle, 8 * (b["n"] + 1)),
                      lane_bytes=lib.ck_alloc_pinned(ctx.handle, (b["total"] if raw else (1 << 16)) + 64),
                      lane_cap=(b["total"] if raw else (1 << 16)), total=C.c_uint64(0))
            rc = lib.ck_pack2_host(b["bytes_p"], b["off_p"], b["n"], pack_flags, threads, ps["dense"], ps["lens"], ps["lane"], ps["lane_bytes"],
                                   ps["lane_cap"], ps["lane_off"], C.byref(ps["total"]))
            if rc != 0:
                raise RuntimeError("ck_pack2_host failed: %d" % rc)
            lt = int(ps["total"].value)
            ps["st"] = N.CkPackedBatch(ps["dense"], b["off_p"], ps["lens"], ps["lane"], ps["lane_bytes"] if lt else None,
                                       ps["lane_off"] if lt else None, lt, b["n"])
            pre_sets.append(ps)

        def pre_step():
            if uniq:
                ctx.uniq_reset()
                if world > 1:
                    dist.barrier()
            for j in range(npre + 1):
                if j < npre:
                    b = batches[j]
                    if uniq:
                        ctx._check(lib.ck_uniq_submit_packed(ctx.handle, j & 1, C.byref(pre_sets[j]["st"]), sub_flags, b["lo"]))
                    else:
                        ctx._check(lib.ck_canon_submit_packed(ctx.handle, j & 1, C.byref(pre_sets[j]["st"]), sub_flags))
                if j >= 1:
                    wait(j - 1)
        pre_step()
        sync_all()
        tp = time.perf_counter()
        for _ in range(e2e_steps):
            pre_step()
        torch.cuda.synchronize()
        dtp = time.perf_counter() - tp
        if world > 1:
            t = torch.tensor([dtp], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dtp = float(t.item())
        pre_cnt = torch.tensor([sum(batches[i]["n"] for i in range(npre))], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(pre_cnt)
        prepacked = {"value": int(pre_cnt.item()) / (dtp / e2e_steps), "unit": "records/s", "records_per_step": int(pre_cnt.item()),
                     "note": "input already packed (ck_pack2_host outside the timed region): H2D of the 2-bit batches + kernels + D2H"}
        for ps in pre_sets:
            for key in ("dense", "lens", "lane", "lane_off", "lane_bytes"):
                lib.ck_free_pinned(ctx.handle, ps[key])
        # leave the first-occurrence state of the full run behind for the parity check below
        e2e_step()
        torch.cuda.synchronize()
    # ---- parity: first indices of the e2e run == the resident run's (global when world > 1)
    parity = None
    if uniq:
        got = np.ctypeslib.as_array(C.cast(out_first_p, C.POINTER(C.c_uint64)), shape=(max(n_mine, 1),))[:n_mine]
        if world > 1:
            allf = [torch.empty(R, dtype=torch.int64, device=dev) for _ in range(world)]
            dist.all_gather(allf, resident_first[:R].contiguous())
            want_all = torch.cat(allf).cpu().numpy().astype(np.uint64)
        else:
            want_all = resident_first[:R].cpu().numpy().astype(np.uint64)
        ok = True
        for i, b in enumerate(batches):
            ok = ok and bool(np.array_equal(got[pos[i]: pos[i + 1]], want_all[b["lo"]: b["lo"] + b["n"]]))
        flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
        if world > 1:
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        parity = bool(int(flag.item()))
        if not parity:
            raise RuntimeError("e2e first_index != resident first_index")
    cnt = torch.tensor([n_mine, sum(b["total"] for b in batches), stats["h2d"]], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(cnt)
    rec_step, bases_step, h2d = int(cnt[0].item()), int(cnt[1].item()), int(cnt[2].item())
    d2h = rec_step * ((8 + 8 + 4) if uniq else (4 + 4 + 1))
    e2e = {"value": rec_step / (dt / e2e_steps), "unit": "records/s", "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": d2h, "steps": e2e_steps, "batches_per_step": len(batches) if world == 1 else n_batches if rounds * world >= n_batches else rounds * world,
           "records_per_batch": RB, "ascii_every": every,
           "ascii_every_probe_seconds": {str(k): round(v, 4) for k, v in probe.items()} if probe else None,
           "api": (("ck_uniq_submit / ck_uniq_wait" if uniq else "ck_canon_submit / ck_canon_wait") if every == 1 else
                   "ck_pack2_host + ck_uniq_submit_packed / ck_uniq_wait" if uniq else "ck_pack2_host + ck_canon_submit_packed / ck_canon_wait")
                  + (" over a peer group (ck_peer_export / ck_peer_attach): global first indices" if world > 1 and uniq else ""),
           "input": "ASCII record bytes + offsets in pinned host memory; the host packer (%d threads per rank) runs INSIDE the timed region%s"
                    % (threads, "; every batch crosses PCIe as ASCII and is normalised / packed on the device (k_prepare): the records of this "
                                "workload are not 2-bit, there is nothing for the host packer to shrink" if every == 1 and raw else
                                "; every batch crosses PCIe as ASCII and is packed on the device (the probe before the timed steps found "
                                "the DMA engine alone faster than any mix with the host packer)" if every == 1 else
                                "; every %d-th batch crosses PCIe as ASCII and is packed on the device instead, so that the DMA engine and the "
                                "packer threads work side by side" % every if every else ""),
           "result": "first_index + hash64 + length per record" if uniq else "start + strand + length per record",
           "gbases_per_s": bases_step / (dt / e2e_steps) / 1e9, "records_per_step": rec_step,
           "host_pack_seconds_per_step_rank0": stats["pack_s"], "first_index_parity_with_resident_run": parity,
           "prepacked": prepacked,
           "note": ("every rank pins its share of the input: the first %d rounds (%d records) of the %d-record input; global uniq over that prefix"
                    % (rounds, rec_step, total_records)) if world > 1 and rec_step < total_records else ""}
    for b in batches:
        lib.ck_free_pinned(ctx.handle, b["bytes_p"]); lib.ck_free_pinned(ctx.handle, b["off_p"])
    for s in sets:
        for key in ("dense", "lens", "lane", "lane_off", "lane_bytes"):
            lib.ck_free_pinned(ctx.handle, s[key])
    for p in (out_first_p, out_hash_p, out_len_p, out_start_p, out_strand_p):
        lib.ck_free_pinned(ctx.handle, p)
    return e2e


SHARDING = {"peer": "partition / query kernels store into the peers' buffers over NVLink (CUDA IPC peer group of the C library, exact counts, device-side barriers)",
            "symm": "the same fused kernels over torch symmetric memory, fixed-capacity buckets",
            "padded": "fixed-capacity buckets, equal-split NCCL all-to-all",
            "exact": "counts, then NCCL all-to-all"}


def make_config(args, w, R, named):
    """`config` of the JSON line: the same dict for the B200 arm and the reference arm"""
    return {"workload": w["desc"] + ("" if named else " [REDUCED: %d records per GPU, not the named config]" % R),
            "records_per_gpu": R, "length_law": ["uniform", "log-uniform"][w["kind"]],
            "length_range": [w["lo"], w["hi"]], "duplicate_fraction": w["dup"] / 1000.0,
            "l2_policy": "inputs larger than L2 (packed arena + ASCII output per step >> 126 MB)",
            "sharding": "contiguous input-index ranges per GPU; uniq keys owned by hash range, exchange: " + SHARDING[args.exchange]}


def _peak():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        return float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def global_first_index_check(ctx, D, torch, dist, dev, rank, world, R, hash_local, first_local):
    """Multi-rank parity of uniq (src/uniq.rs:42-78: ONE `seen` map over the whole input): every rank's hashes and the
    first indices the fused exchange gave it are gathered on rank 0, which rebuilds the global first-occurrence index with the
    single-GPU table (ck_dev_table_insert / ck_dev_table_first -- the path the oracle tests pin) over all world * R keys in
    input order and compares.  -> (parity ok, global unique records) on rank 0, (None, None) elsewhere."""
    hs = [torch.empty(R, dtype=torch.int64, device=dev) for _ in range(world)] if rank == 0 else None
    fs = [torch.empty(R, dtype=torch.int64, device=dev) for _ in range(world)] if rank == 0 else None
    dist.gather(hash_local[:R].contiguous(), hs, dst=0)
    dist.gather(first_local[:R].contiguous(), fs, dst=0)
    if rank != 0:
        return None, None
    table = D.DeviceTable(ctx, capacity_keys=int(R * world * 1.05) + 1024, dev=dev)
    slots = [torch.empty(R, dtype=torch.int64, device=dev) for _ in range(world)]
    for r in range(world):
        table.insert(hs[r], R, slots[r], base_index=r * R)
    ok, uniq = True, 0
    want = torch.empty(R, dtype=torch.int64, device=dev)
    for r in range(world):
        table.first(slots[r], R, want)
        ok = ok and bool(torch.equal(want, fs[r]))
        uniq += int((want == torch.arange(r * R, (r + 1) * R, device=dev)).sum().item())
    return ok, uniq


def b200_arm(args, wname, R, rank, local_rank, world, dev, steps, warmup, want_e2e, want_cpu, scaling, dump_prefix=""):
    """One workload on this rank's shard of R records: resident measurement (value, roofline), optional e2e and CPU legs.
    With --dump-outputs, rank 0 writes its shard's results of the last timed step as <dump_prefix><name>.npy.
    Returns the JSON line as a dict on rank 0 (None elsewhere)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    import circkit_b200
    from circkit_b200 import device as D
    from circkit_b200 import exchange as X

    w = dict(WORKLOADS[wname])
    seed = SEEDS[wname]
    named = R == w["records"] or scaling == "strong"
    metric = "canonicalize+uniq records/sec" if w["uniq"] else "canonicalize records/sec"
    config = make_config(args, w, R, named)
    w["mask"] = D.class_mask_for(w["lo"], w["hi"])
    e2e_on = want_e2e
    ctx = circkit_b200.Context(device=local_rank, max_batch_bytes=(256 << 20) if e2e_on else 0,
                               max_batch_records=(1 << 20) if e2e_on else 0,
                               table_capacity=R if (w["uniq"] and e2e_on) else 0)
    sampler = ClockSampler(local_rank)                     # started early: nvidia-smi needs ~100 ms to come up
    sampler.start()
    base_index = rank * R
    raw_dev = None
    if w.get("raw"):
        # config 3: raw record bytes resident in HBM (numpy generator circkit_b200/synth_host.py, 500 k distinct records tiled to
        # the requested count -- generating 5 M on the host would take minutes); every symbol lane is exercised:
        # normalise + classify + pack + canonicalise per step
        from circkit_b200 import synth_host
        tile_n = min(R, 500_000)
        a_np, o_np = synth_host.make_iupac_records(tile_n, w["lo"], w["hi"], seed + rank)
        reps = (R + tile_n - 1) // tile_n
        a_t = torch.from_numpy(a_np).to(dev)
        l_t = torch.from_numpy((o_np[1:] - o_np[:-1]).astype(np.int64)).to(dev)
        raw_dev = a_t.repeat(reps)
        lens_all = l_t.repeat(reps)[:R]
        offs = torch.zeros(R + 1, dtype=torch.int64, device=dev)
        torch.cumsum(lens_all, 0, out=offs[1:])
        total_raw = int(offs[-1].item())
        raw_dev = raw_dev[:total_raw].contiguous()
        batch = D.DeviceBatch(offs, None, R, total_raw)
        lens_out = torch.empty(R, dtype=torch.int32, device=dev)
        ws = D.Workspace(ctx, R, total_raw, dev)
        w["mask"] = 0
    else:
        batch = D.synth_batch(ctx, seed=seed, first_index=base_index, n_records=R, kind=w["kind"], lo=w["lo"], hi=w["hi"],
                              dup_permille=w["dup"], adversarial_permille=w["adv"], device=dev)
        ws = D.Workspace(ctx, R, 0, dev)
    outs = D.CanonOutputs(R, batch.total, dev, want_bytes=True, want_hash=w["uniq"], aligned=True)
    lens = batch.lens
    if w["uniq"]:
        table = D.DeviceTable(ctx, capacity_keys=int(R * 1.05) + 1024, dev=dev)   # owns ~R keys of the global set
        first = torch.empty(R, dtype=torch.int64, device=dev)
        slot_cache = {}

        def first_fn(h, idx):
            m = h.numel()
            if m not in slot_cache:
                slot_cache[m] = (torch.empty(max(m, 1), dtype=torch.int64, device=dev),
                                 torch.empty(max(m, 1), dtype=torch.int64, device=dev))
            slots, out = slot_cache[m]
            table.insert(h, m, slots, index=idx, base_index=base_index if idx is None else 0)
            table.first(slots, m, out)
            return out[:m]

        def insert_pairs_fn(pairs):                 # owner side, phase 1: returns the slots for the later query
            m = pairs.shape[0]
            slots = torch.empty(max(m, 1), dtype=torch.int64, device=dev)
            table.insert_pairs(pairs, m, slots)
            return slots

        def first_query_fn(slots, m):               # owner side, phase 2
            out = torch.empty(max(m, 1), dtype=torch.int64, device=dev)
            table.first(slots, m, out)
            return out[:m]

        def first_pairs_fn(pairs):                  # owner side of the padded exchange: insert, then query, padding skipped
            m = pairs.shape[0]
            key = ("pairs", m)
            if key not in slot_cache:
                slot_cache[key] = (torch.empty(max(m, 1), dtype=torch.int64, device=dev),
                                   torch.empty(max(m, 1), dtype=torch.int64, device=dev))
            slots, out = slot_cache[key]
            table.insert_pairs(pairs, m, slots)
            table.first(slots, m, out)
            return out[:m]

    padded = {"on": world > 1 and args.exchange in ("symm", "padded") and w["uniq"], "overflow": torch.zeros(1, dtype=torch.int32, device=dev),
              "peer": None}
    peer_group = None
    if world > 1 and w["uniq"] and args.exchange == "peer":
        # the library's own peer group (CUDA IPC).  If any rank cannot set it up, every rank takes the NCCL buckets instead and
        # the JSON line says so
        why = ""
        try:
            peer_group = D.PeerGroup(ctx, max(R, ctx.max_batch_records, 1), world, rank)
            ctx._peer_attached = True
        except Exception as e:                              # noqa: BLE001 -- reported, not hidden
            why = "%s: %s" % (type(e).__name__, str(e).splitlines()[0] if str(e) else "")
        okt = torch.tensor([1 if peer_group is not None else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        if not int(okt.item()):
            peer_group = None
            padded["on"] = True
            config["sharding"] += " [peer group unavailable on this node (%s): fixed-capacity buckets through NCCL instead]" % (why or "another rank")
    if padded["on"] and args.exchange == "symm":
        peer, why = None, ""
        try:
            peer = D.PeerExchange(ctx, R, world, rank, dev)
        except Exception as e:                              # noqa: BLE001 -- reported, not hidden
            why = "%s: %s" % (type(e).__name__, str(e).splitlines()[0] if str(e) else "")
        okt = torch.tensor([1 if peer is not None else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        if int(okt.item()):
            padded["peer"] = peer
        else:
            config["sharding"] += " [symmetric memory unavailable on this node (%s): fixed-capacity buckets through NCCL instead]" % (why or "another rank")
    stage_stream, outs_sets, first_sets, pipe, partitioner = None, None, None, None, None
    if w["uniq"] and raw_dev is None:
        overlap = args.overlap if args.overlap is not None else world > 1
        slots_1gpu = torch.empty(max(R, 1), dtype=torch.int64, device=dev) if world == 1 else None
        stage_stream = torch.cuda.Stream(device=dev) if overlap else None
        config["pipelining"] = ("table / exchange stage of step k on a second stream, overlapping the kernels of step k + 1 (double-buffered outputs)"
                                if overlap else "none: every step's stages in stream order")
        outs_sets = [outs, D.CanonOutputs(R, batch.total, dev, want_bytes=True, want_hash=True, aligned=True) if overlap else outs]
        first_sets = [first, torch.empty_like(first) if overlap else first]
        pipe = dict(k=0, done=[torch.cuda.Event(), torch.cuda.Event()], canon=[torch.cuda.Event(), torch.cuda.Event()])
        partitioner = D.OwnerPartitioner(ctx, R, world, dev) if world > 1 else None

    def step():
        if raw_dev is not None:
            D.canon_bytes(ctx, raw_dev, batch.offsets, R, batch.total, outs, lens_out, ws, normalize=True)
            return
        if not w["uniq"]:
            D.canon_packed2(ctx, batch, outs, ws, class_mask=w["mask"])
            return
        # uniq: kernels of step k on the current stream into output set k & 1; its table / exchange stage on `stage_stream`
        # with --overlap (else the same stream), so that it overlaps the kernels of step k + 1
        i = pipe["k"] & 1
        pipe["k"] += 1
        o_i, f_i = outs_sets[i], first_sets[i]
        cur = torch.cuda.current_stream()
        if world == 1 and stage_stream is None:
            # one GPU: canonicalise + hash, then the table passes, straight into this step's result buffer
            D.canon_packed2(ctx, batch, o_i, ws, class_mask=w["mask"])
            table.clear()
            table.insert(o_i.hash[:R], R, slots_1gpu, base_index=base_index)
            table.first(slots_1gpu, R, f_i)
            return
        cur.wait_event(pipe["done"][i])             # the stage of step k - 2 has finished with this output set
        D.canon_packed2(ctx, batch, o_i, ws, class_mask=w["mask"])
        pipe["canon"][i].record(cur)
        st = stage_stream if stage_stream is not None else cur
        with torch.cuda.stream(st):
            st.wait_event(pipe["canon"][i])
            table.clear()
            if world == 1:
                table.insert(o_i.hash[:R], R, slots_1gpu, base_index=base_index)
                table.first(slots_1gpu, R, f_i)
            elif peer_group is not None:            # exact counts, no padding, nothing to check afterwards
                peer_group.first_index(o_i.hash[:R], base_index, table, f_i)
            elif padded["on"]:
                # fixed-capacity buckets: no counts to exchange, no host synchronisation in the step; an overflowing bucket is
                # flagged on the device and checked after the steps have been queued
                if padded["peer"] is not None:      # partition and query kernels store straight into the peers' buffers
                    state = padded["peer"].first_index(o_i.hash[:R], base_index, table, f_i)
                else:                               # the same buckets through one equal-split all-to-all each way
                    f, state = X.exchange_first_index_padded(o_i.hash[:R], base_index, first_pairs_fn, padded_fn=partitioner.padded)
                    f_i.copy_(f)
                padded["overflow"].add_(state[world: world + 1])
            else:
                pend = X.exchange_send(o_i.hash[:R], base_index, partitioner, insert_pairs_fn)
                f_i.copy_(X.exchange_finish(pend, first_query_fn))
            pipe["done"][i].record(st)

    def drain():
        if stage_stream is not None:
            torch.cuda.current_stream().wait_stream(stage_stream)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    t_window0 = time.time()
    for _ in range(warmup):
        step()
    drain()
    sync_all()
    D.check(ctx, ws)
    if padded["on"]:
        ov = padded["overflow"].clone().to(torch.int64)
        dist.all_reduce(ov, op=dist.ReduceOp.MAX)
        if int(ov.item()):                              # a bucket overflowed somewhere: every rank takes the exact path
            padded["on"] = False
            padded["peer"] = None
            padded["overflow"].zero_()
            config["sharding"] += " [a fixed-capacity bucket overflowed in the warm-up: exact-count exchange instead]"
            for _ in range(warmup):
                step()
            drain()
            sync_all()
    ctx._lib.ck_kernel_timing(ctx.handle, 1)
    D.kernel_times(ctx)
    launches0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record()
    for _ in range(steps):
        step()
    drain()
    e1.record()
    sync_all()
    ms = e0.elapsed_time(e1)
    if padded["on"] and int(padded["overflow"].item()):
        raise RuntimeError("padded exchange overflowed inside the timed steps although the warm-up steps on the same data did not")
    if pipe is not None:
        first = first_sets[(pipe["k"] - 1) & 1]             # result of the last step
        outs_last = outs_sets[(pipe["k"] - 1) & 1]
    else:
        outs_last = outs
    clocks = sampler.stop(t_window0, time.time())
    launches = ctx.launch_count() - launches0
    ktimes = D.kernel_times(ctx)
    ctx._lib.ck_kernel_timing(ctx.handle, 0)
    D.check(ctx, ws)
    if args.dump_outputs and rank == 0:
        per_record = {"length": lens_out if raw_dev is not None else lens, "start": outs_last.start, "strand": outs_last.strand}
        if outs_last.hash is not None:
            per_record["hash"] = outs_last.hash
        if w["uniq"]:
            per_record["first_index"] = first
        dump_outputs(args.dump_outputs, dump_prefix, R, per_record, canon=(outs_last.out, batch.offsets))
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms_per_step = ms / steps
    total_records = R * world
    total_bases = batch.total
    if world > 1:
        tb = torch.tensor([batch.total], dtype=torch.int64, device=dev)
        dist.all_reduce(tb)
        total_bases = int(tb.item())
    value = total_records / (ms_per_step / 1e3)

    # ---------------- multi-rank parity: the global first-occurrence index, rebuilt on rank 0 with the single-GPU table
    global_parity, global_unique = None, None
    if w["uniq"]:
        if world > 1:
            global_parity, global_unique = global_first_index_check(ctx, D, torch, dist, dev, rank, world, R, outs_last.hash, first)
            flag = torch.tensor([1 if (rank != 0 or global_parity) else 0], dtype=torch.int32, device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if not int(flag.item()):
                raise RuntimeError("multi-rank uniq: first indices of the exchange differ from the single-table rebuild on rank 0")
        else:
            global_unique = int((first == torch.arange(base_index, base_index + R, device=dev)).sum().item())

    # ---------------- roofline of the dominant kernel (rank 0's launches)
    from circkit_b200.device import CLASS_NAMES
    # (the small per-class launches run side by side on forked streams: the interval of a launch with no records can be as
    # long as the kernel it waited behind, so only classes that hold records of this batch are candidates)
    byte_ranges = {"4bit_lane_129_2048": (129, 2048), "4bit_le_2048": (1, 2048), "4bit_le_212992": (2049, 212992), "byte_le_1024": (1, 1024), "byte_le_106496": (1025, 106496)}

    def holds_records(c):
        lo_c, hi_c = D.CLASS_RANGE.get(c) or byte_ranges.get(c, (0, 0))
        if (c in byte_ranges) != bool(w.get("raw")):
            return False
        return bool(((lens >= lo_c) & (lens <= hi_c)).any())
    dom = max((c for c in CLASS_NAMES if ktimes[c][1] and holds_records(c) and not c.startswith("table")), key=lambda c: ktimes[c][0])
    lo_n, hi_n = D.CLASS_RANGE.get(dom, (1, 1 << 40))
    byte_lane = dom.startswith(("4bit", "byte"))
    # bytes this kernel's launch moves by the algorithm: packed read + ASCII write + 16 (+8 hash write);
    # the table's 32 B/record belong to the table kernels, not to this launch
    sel = lens[(lens >= lo_n) & (lens <= hi_n)]
    if byte_lane:        # byte lanes: n bytes read + n bytes written + 16 (SURVEY 8d); every record of the batch charged to the lane
        alg_bytes = int((2 * sel + 16).sum().item())
    else:
        alg_bytes = int((8 * ((sel + 31) // 32) + sel + 16 + (8 if w["uniq"] else 0)).sum().item())
    launches_per_step = max(ktimes[dom][1], 1) / steps
    dom_ms = ktimes[dom][0] / steps                                   # per step: all launches of the dominant kernel
    peak, peak_src = _peak()
    achieved = alg_bytes / (dom_ms / 1e3) / 1e9 if dom_ms > 0 else 0.0
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            traffic = tj.get(wname, {}).get(dom)
            if traffic is not None:
                traffic = int(traffic / launches_per_step)
                traffic_src = "ncu --set full, separate run (%s)" % tj.get("_source", "profiles/")
        except Exception:
            traffic = None
    kernel_share = {c: round(ktimes[c][0] / steps, 4) for c in CLASS_NAMES if ktimes[c][1]}
    roofline = {"bound": "hbm", "kernel": "%s [%s]" % ("k_canon_seg (warp per record, a lane per segment, 16-mer keys)" if "seg" in dom else "k_canon_cta<2>" if "65536" in dom or "425984" in dom else "k_canon_l4 (lane per record, 4-bit strands packed by k_pack4)" if dom.startswith("4bit_lane") else "k_canon_warp (byte-level lane)" if byte_lane else "k_canon_s2 (lane per record, single-copy arena, 128-bit loads)" if getattr(batch, "single", False) else "k_canon_s3 (lane per record, doubled arena, 256-bit loads)", dom),
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": int(alg_bytes / launches_per_step),
                "kernel_ms_per_launch": dom_ms / launches_per_step, "launches_per_step": launches_per_step,
                "frac_of_nominal_8TBs": achieved / 8000.0, "class_kernel_ms_per_step": kernel_share,
                "step_ms": ms_per_step}

    if w.get("raw"):
        roofline["note"] = ("the layout passes in front of this kernel -- k_prepare (normalise + classify + pack) and k_pack4 (4-bit strands) -- "
                            "are timed in class_kernel_ms_per_step as 'prepare' and 'pack4': each of them takes longer than the "
                            "canonicalisation kernel the roofline is quoted for")
    # ---------------- e2e through the host-buffer C ABI (pinned host memory, copies timed)
    e2e = None
    if want_e2e:
        e2e = e2e_leg(args, ctx, D, torch, dist, dev, rank, world, w, wname, R, first if w["uniq"] else None, sync_all, steps)

    # ---------------- CPU baseline beside it (rank 0, N = 1)
    cpu = None
    if rank == 0 and world == 1 and want_cpu:
        r = cpu_arm(w, seed, args.cpu_seconds, 3, 1, w["uniq"])
        cpu = {"value": r["records_per_s"], "unit": "records/s", "cores": r["cores"], "kind": "port",
               "gbases_per_s": r["gbases_per_s"],
               "sample": "%d records / %.1f Mbases of the same length law and duplicate rate (independent numpy draw), "
                         "worker stage on %d threads + serial consumer, step = max of the two; O(1)-indexed Duval "
                         "(conservative)" % (r["sample_records"], r["sample_bases"] / 1e6, r["cores"]),
               "faithful_cost_footnote": cpu_faithful_footnote(w, seed)}

    line = None
    if rank == 0:
        line = {"metric": metric, "value": value, "unit": "records/s", "n_gpus": world, "steps": steps,
                "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling,
                "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config,
                "gbases_per_s": total_bases / (ms_per_step / 1e3) / 1e9, "clocks": clocks, "e2e": e2e,
                "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
                "global_unique_records": global_unique, "global_parity": global_parity,
                "global_parity_how": ("every rank's hash64 + first_index gathered on rank 0; first index rebuilt over all %d keys "
                                      "with the single-GPU table and compared" % total_records) if world > 1 and w["uniq"] else None}
    ctx.close()
    del batch, outs, ws
    if w["uniq"]:
        del table, first, outs_sets, first_sets
    torch.cuda.empty_cache()
    return line


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.workload == "mono":
        if rank == 0:
            (bench_monomerize_reference if args.impl == "reference" else bench_monomerize)(args)
        return

    # ---------------- reference arm: the CPU path, rank 0 only
    if args.impl == "reference":
        if rank != 0:
            return
        w = dict(WORKLOADS[args.workload])
        seed = SEEDS[args.workload]
        if args.records:
            w["records"] = args.records
        metric = "canonicalize+uniq records/sec" if w["uniq"] else "canonicalize records/sec"
        r = cpu_arm(w, seed, max(args.cpu_seconds, 4.0 * (args.steps + args.warmup)), args.steps, args.warmup, w["uniq"])
        sample = ("oracle port of circKit's path (Duval x2 + revcomp + compare, xxh3, keep-first map; O(1) byte "
                  "indexing -- conservative: the reference's chars().nth(i) is O(i)); a bounded SAMPLE of %d records / %.1f Mbases of the "
                  "workload per step (a rate, not the %d records of the named config), worker stage on %d threads, consumer stage "
                  "serial, step = max of the two" % (r["sample_records"], r["sample_bases"] / 1e6, w["records"], r["cores"]))
        config = make_config(args, w, w["records"], not args.records)
        line = {"impl": "reference", "metric": metric, "value": r["records_per_s"], "unit": "records/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": config, "gbases_per_s": r["gbases_per_s"],
                "cpu_baseline": {"value": r["records_per_s"], "unit": "records/s", "cores": r["cores"], "kind": "port",
                                 "sample": sample},
                "e2e": {"value": r["records_per_s"], "unit": "records/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "reference_sample": {"records_per_step": r["sample_records"], "bases_per_step": r["sample_bases"],
                                     "note": "each step is a bounded sample of the workload: the value is a rate"},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    # ---------------- B200 arm
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    R = args.records or WORKLOADS[args.workload]["records"]
    line = b200_arm(args, args.workload, R, rank, local_rank, world, dev, args.steps, args.warmup,
                    want_e2e=not args.no_e2e, want_cpu=not args.no_cpu, scaling="weak")
    # ---------------- config 5 as the north star states it: ONE 100 M-record uniq split over the N GPUs (strong scaling),
    # reported as a sub-record of the same line
    if args.workload == "c2" and not args.no_config5 and not args.records:
        total5 = args.c5_records
        R5 = total5 // world
        sub = b200_arm(args, "c5", R5, rank, local_rank, world, dev, max(2, min(args.steps, 5)), 3,
                       want_e2e=False, want_cpu=False, scaling="strong", dump_prefix="config5_")
        if rank == 0:
            line["config5"] = {k: sub[k] for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "scaling",
                                                    "gbases_per_s", "gpu_launches", "global_unique_records", "global_parity")}
            line["config5"]["records_total"] = R5 * world
            line["config5"]["records_per_gpu"] = R5
            line["config5"]["workload"] = "config 5: uniq over %d viroid-length records (250-400 nt, 30%% duplicates), split over %d GPU(s)" % (R5 * world, world)
            line["config5"]["roofline"] = {k: sub["roofline"][k] for k in ("kernel", "achieved", "peak", "frac", "kernel_ms_per_launch", "class_kernel_ms_per_step")}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
