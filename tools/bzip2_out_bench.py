"""The device bzip2 encoder and the CLI's `-o out.fa.bz2` on two FASTA files (one GPU).

    python tools/bzip2_out_bench.py --out DIR [--parent TREE] [--records 1000000] [--dup-records 60000]

Files (in a temporary directory), as tools/gzip_out_bench.py writes them:
  mono  bench.py's `--workload mono` shape, written by tools/mono_stream_bench.write_fasta (1 M records, 767 MB)
  dup   60 k records of 200-1200 random A/C/G/T with 70-column lines; 30 % are copies of one of the previous 50 (seeded)
Reports one JSON line per measurement, with the card's name and power limit read in the same run:
  (a) encoder    ck_bzip2_submit / ck_bzip2_wait per call of up to 64 MiB (each call given the previous call's unconsumed
                 tail), timed by CUDA events after a warm-up call, in GB/s of input; the per-stage device time (RLE1 and
                 cuts, BWT, MTF, tables, pack) from ck_bzip2_stats and the BWT's sort rounds; the stream is compared byte
                 for byte with bz2.compress(file, 9)
  (b) cli        wall time of `canonicalize in.fa -o out.fa`, of `-o out.fa.bz2` with this tree, of `-o out.fa.bz2` with the
                 --parent tree (host BZ2File), and of `-o out.fa` once more; the two .bz2 files are compared byte for byte
                 with each other and with bz2.compress of the plain output.
"""
from __future__ import annotations

import argparse
import bz2
import json
import os
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

STAGES = ("rle1_cuts", "bwt", "mtf", "tables", "pack")


def encoder(path: str, info: dict) -> dict:
    import numpy as np
    import torch
    from circkit_b200 import Context, cli, _native as N
    data = open(path, "rb").read()
    ctx = Context(max_batch_bytes=0, max_batch_records=0)
    step = N.CK_BZIP2_MAX_BYTES
    ctx.bzip2(data[:step], True)                                   # warm-up: allocation, module load
    parts, tail, pos, bits, nbits, crc, ms, calls, rounds = [cli.BZIP2_HEADER], b"", 0, 0, 0, 0, 0.0, 0, []
    stage = [0.0] * len(STAGES)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    while True:
        take = step - len(tail)
        buf = tail + data[pos:pos + take]
        pos += take
        final = pos >= len(data)
        src = np.frombuffer(buf, dtype=np.uint8)
        t0.record()
        ctx.bzip2_submit(0, src, final, bits, nbits, crc)
        out, consumed, bits, nbits, crc = ctx.bzip2_wait(0)
        t1.record()
        t1.synchronize()
        ms += t0.elapsed_time(t1)
        st, r = ctx.bzip2_stats(0)
        stage = [a + b for a, b in zip(stage, st)]
        rounds.append(r)
        calls += 1
        parts.append(out)
        tail = buf[consumed:]
        if final:
            break
    v = (bits << 80 | cli.BZIP2_EOS << 32 | crc) << (-(nbits + 80) % 8)
    parts.append(v.to_bytes((nbits + 87) // 8, "big"))
    dev = b"".join(parts)
    ref = bz2.compress(data, 9)
    ctx.close()
    return {"input_bytes": len(data), "device_bytes": len(dev), "libbz2_bytes": len(ref), "identical": dev == ref,
            "ratio": len(dev) / len(data), "calls": calls, "device_ms": ms, "device_gb_per_s": len(data) / ms / 1e6,
            "stage_ms": dict(zip(STAGES, stage)), "bwt_rounds": rounds, **info}


def run_cli(tree: str, src: str, dst: str) -> float:
    import time
    env = dict(os.environ, PYTHONPATH=tree)
    t0 = time.perf_counter()
    subprocess.run([sys.executable, "-m", "circkit_b200", "canonicalize", src, "-o", dst], cwd=tree, env=env, check=True)
    return time.perf_counter() - t0


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True)
    ap.add_argument("--parent", help="source tree whose CLI writes .bz2 on the host (built in place)")
    ap.add_argument("--records", type=int, default=1_000_000)
    ap.add_argument("--dup-records", type=int, default=60_000)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    import __graft_entry__
    __graft_entry__.build()
    if args.parent:
        subprocess.run([sys.executable, "-c", "import __graft_entry__ as g; g.build()"], cwd=args.parent, check=True)
    from gzip_out_bench import write_dup_fasta
    from mono_stream_bench import gpu_info, write_fasta
    info = gpu_info()
    tmp = tempfile.mkdtemp(prefix="bzip2_out_bench_")
    lines = []
    try:
        files = {"mono": os.path.join(tmp, "mono.fa"), "dup": os.path.join(tmp, "dup.fa")}
        write_fasta(files["mono"], args.records)
        write_dup_fasta(files["dup"], args.dup_records)
        for name, path in files.items():
            line = {"run": "encoder", "file": name, **encoder(path, info)}
            print(json.dumps(line), flush=True)
            lines.append(line)
        for name, path in files.items():
            plain = os.path.join(tmp, "o.fa")
            line = {"run": "cli", "file": name, "input_mb": os.path.getsize(path) / 1e6, "plain_s": run_cli(ROOT, path, plain)}
            want = bz2.compress(open(plain, "rb").read(), 9)
            line["bz2_s"] = run_cli(ROOT, path, os.path.join(tmp, "o.fa.bz2"))
            got = open(os.path.join(tmp, "o.fa.bz2"), "rb").read()
            line["bz2_identical"] = got == want
            line["bz2_bytes"] = len(got)
            if args.parent:
                line["parent_bz2_s"] = run_cli(args.parent, path, os.path.join(tmp, "p.fa.bz2"))
                line["parent_bz2_identical"] = open(os.path.join(tmp, "p.fa.bz2"), "rb").read() == got
            line["plain_again_s"] = run_cli(ROOT, path, plain)     # the first run of a file also warms the page cache
            line["bz2_over_plain"] = line["bz2_s"] / min(line["plain_s"], line["plain_again_s"])
            line.update(info)
            print(json.dumps(line), flush=True)
            lines.append(line)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    with open(os.path.join(args.out, "bzip2_out_bench.jsonl"), "w") as f:
        f.write("".join(json.dumps(x) + "\n" for x in lines))
    ok = all(x.get("identical", True) and x.get("bz2_identical", True) and x.get("parent_bz2_identical", True)
             for x in lines)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
