"""The device DEFLATE encoder and the CLI's `-o out.fa.gz` on two FASTA files (one GPU).

    python tools/gzip_out_bench.py --out DIR [--parent TREE] [--records 1000000] [--dup-records 60000]

Files (in a temporary directory):
  mono  bench.py's `--workload mono` shape, written by tools/mono_stream_bench.write_fasta (1 M records, 767 MB)
  dup   60 k records of 200-1200 random A/C/G/T with 70-column lines and headers like `>sample_3|read_000123 len=745 cov=12.5`;
        30 % of the records are copies of one of the previous 50 (seeded)
Reports one JSON line per measurement, with the card's name and power limit read in the same run:
  (a) encoder    ck_deflate_submit / ck_deflate_wait per 64 MiB call of the file (each call given the 32 KiB before it),
                 timed by CUDA events after a warm-up call, in GB/s of input; the device's size and zlib's level-1 and
                 level-6 sizes of the same bytes (one raw deflate stream over the whole file), and their ratios
  (b) cli        wall time of `canonicalize in.fa -o out.fa`, of `-o out.fa.gz` with this tree, of `-o out.fa.gz` with
                 the --parent tree (host gzip), and of `-o out.fa` once more; the decompressed outputs are compared byte
                 for byte with the plain one.
"""
from __future__ import annotations

import argparse
import gzip
import json
import os
import random
import shutil
import subprocess
import sys
import tempfile
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def write_dup_fasta(path: str, n: int, seed: int = 5) -> int:
    rng = random.Random(seed)
    recs = []
    with open(path, "wb") as f:
        for i in range(n):
            if recs and rng.random() < 0.3:
                body = rng.choice(recs[-50:])
            else:
                body = rng.randbytes(rng.randint(200, 1200)).translate(bytes(b"ACGT"[k & 3] for k in range(256)))
                recs.append(body)
            head = b">sample_%d|read_%06d len=%d cov=%.1f\n" % (rng.randrange(8), i, len(body), rng.uniform(1, 60))
            f.write(head + b"\n".join(body[k:k + 70] for k in range(0, len(body), 70)) + b"\n")
    return os.path.getsize(path)


def encoder(path: str, info: dict) -> dict:
    import numpy as np
    import torch
    from circkit_b200 import Context, _native as N
    data = open(path, "rb").read()
    ctx = Context(max_batch_bytes=0, max_batch_records=0)
    step = N.CK_DEFLATE_MAX_BYTES
    src = np.frombuffer(data, dtype=np.uint8)
    ctx.deflate(src[:step])                                       # warm-up: allocation, module load
    parts, crc, ms = [], 0, 0.0
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for lo in range(0, len(data), step):
        d = data[max(0, lo - 32768):lo]
        t0.record()
        ctx.deflate_submit(0, src[lo:lo + step], d, crc)
        out, crc = ctx.deflate_wait(0)
        t1.record()
        t1.synchronize()
        ms += t0.elapsed_time(t1)
        parts.append(out)
    dev = b"".join(parts)
    assert zlib.decompressobj(-15).decompress(dev) == data and crc == zlib.crc32(data)
    sizes = {}
    for lvl in (1, 6):
        c = zlib.compressobj(lvl, zlib.DEFLATED, -15)
        sizes[lvl] = len(c.compress(data) + c.flush())
    ctx.close()
    return {"input_bytes": len(data), "device_bytes": len(dev), "zlib1_bytes": sizes[1], "zlib6_bytes": sizes[6],
            "device_ratio": len(dev) / len(data), "device_over_zlib6": len(dev) / sizes[6],
            "device_over_zlib1": len(dev) / sizes[1], "calls": len(parts), "device_ms": ms,
            "device_gb_per_s": len(data) / ms / 1e6, **info}


def run_cli(tree: str, src: str, dst: str) -> float:
    env = dict(os.environ, PYTHONPATH=tree)
    t0 = time.perf_counter()
    subprocess.run([sys.executable, "-m", "circkit_b200", "canonicalize", src, "-o", dst], cwd=tree, env=env, check=True)
    return time.perf_counter() - t0


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True)
    ap.add_argument("--parent", help="source tree whose CLI writes .gz on the host (built in place)")
    ap.add_argument("--records", type=int, default=1_000_000)
    ap.add_argument("--dup-records", type=int, default=60_000)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    import __graft_entry__
    __graft_entry__.build()
    if args.parent:
        subprocess.run([sys.executable, "-c", "import __graft_entry__ as g; g.build()"], cwd=args.parent, check=True)
    from mono_stream_bench import gpu_info, write_fasta
    info = gpu_info()
    tmp = tempfile.mkdtemp(prefix="gzip_out_bench_")
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
            want = open(plain, "rb").read()
            line["gz_s"] = run_cli(ROOT, path, os.path.join(tmp, "o.fa.gz"))
            line["gz_identical"] = gzip.decompress(open(os.path.join(tmp, "o.fa.gz"), "rb").read()) == want
            line["gz_bytes"] = os.path.getsize(os.path.join(tmp, "o.fa.gz"))
            if args.parent:
                line["parent_gz_s"] = run_cli(args.parent, path, os.path.join(tmp, "p.fa.gz"))
                line["parent_gz_identical"] = gzip.decompress(open(os.path.join(tmp, "p.fa.gz"), "rb").read()) == want
                line["parent_gz_bytes"] = os.path.getsize(os.path.join(tmp, "p.fa.gz"))
            line["plain_again_s"] = run_cli(ROOT, path, plain)     # the first run of a file also warms the page cache
            line["gz_over_plain"] = line["gz_s"] / min(line["plain_s"], line["plain_again_s"])
            line.update(info)
            print(json.dumps(line), flush=True)
            lines.append(line)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    with open(os.path.join(args.out, "gzip_out_bench.jsonl"), "w") as f:
        f.write("".join(json.dumps(x) + "\n" for x in lines))
    ok = all(x.get("gz_identical", True) and x.get("parent_gz_identical", True) for x in lines)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
