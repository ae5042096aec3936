"""`python -m circkit_b200 uniq` from stdin past the size of a fixed table: the uniq table starts at cli.UNIQ_TABLE_KEYS keys
and has to grow on the device as the distinct records arrive (one GPU).

    python tools/uniq_growth_bench.py --out DIR [--records 25200000] [--parent TREE]

Writes --records distinct single-line records ('>' 8-digit id '\\n' 32 random bases '\\n', 43 bytes each, seeded) to a
temporary file and runs `python -m circkit_b200 uniq -o OUT < FILE`.  Every record is distinct, so without -c the output
must equal the input byte for byte.  (A table of 2^24 keys, the size the CLI used to give stdin input, holds 25 165 840 of
them at most.)  Then the same file goes through the library as the CLI drives it (text batches on alternating slots), with
ck_uniq_table_info read after every submit: the growths, the final capacity, and the submit time of each growth against the
median submit.  --parent TREE: the CLI of another source tree (built in place) on the same input, for its exit code.
Prints one JSON line per step, with the card's name and power limit read in the same process.
"""
from __future__ import annotations

import argparse
import filecmp
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.splitlines()[0].split(", ") + ["?"])[:2] if q.returncode == 0 and q.stdout else ("?", "?")
    return {"gpu": name.strip(), "power_limit": power.strip()}


def write_records(path: str, n: int, seed: int = 11) -> int:
    rng = np.random.default_rng(seed)
    letters = np.frombuffer(b"ACGT", np.uint8)
    with open(path, "wb") as f:
        for lo in range(0, n, 1 << 20):
            hi = min(n, lo + (1 << 20))
            a = np.empty((hi - lo, 43), dtype=np.uint8)
            ids = np.arange(lo, hi, dtype=np.int64)
            a[:, 0] = ord(">")
            for d in range(8):
                a[:, 1 + d] = 48 + (ids // 10 ** (7 - d)) % 10
            a[:, 9] = a[:, 42] = ord("\n")
            a[:, 10:42] = letters[rng.integers(0, 4, (hi - lo, 32))]
            f.write(a.tobytes())
    return os.path.getsize(path)


def run_cli(tree: str, src: str, dst: str) -> dict:
    env = dict(os.environ, PYTHONPATH=tree)
    t0 = time.perf_counter()
    with open(src, "rb") as stdin:
        p = subprocess.run([sys.executable, "-m", "circkit_b200", "uniq", "-o", dst], cwd=tree, env=env, stdin=stdin,
                           capture_output=True, text=True)
    return {"exit": p.returncode, "wall_s": time.perf_counter() - t0, "stderr": p.stderr.strip()[-300:]}


def growth_trace(src: str) -> dict:
    """the file through the library as cli._Pump drives it, with the table read after every submit"""
    sys.path.insert(0, ROOT)
    from circkit_b200 import cli
    ctx = cli._context(cli.UNIQ_TABLE_KEYS)
    ctx.uniq_grow()
    text = open(src, "rb").read()
    cap0 = ctx.table_info()[1]
    submits, grows_at, pend, base = [], [], None, 0
    try:
        for b, (lo, hi) in enumerate(cli._text_batches(text, cli.MAX_BATCH_BYTES, cli.MAX_BATCH_RECORDS)):
            slot = b & 1
            before = ctx.table_info()                     # synchronises both slots: the submit below starts from idle
            t0 = time.perf_counter()
            n = ctx.fasta_submit(slot, memoryview(text)[lo:hi], "uniq", base_index=base)
            dt = time.perf_counter() - t0
            after = ctx.table_info()
            submits.append(dt)
            if after[2] > before[2]:
                grows_at.append({"batch": b, "keys_before": before[0], "capacity_before": before[1], "capacity_after": after[1],
                                 "submit_s": dt})
            if pend is not None:
                ctx.fasta_wait(pend)
            pend, base = slot, base + n
        ctx.fasta_wait(pend)
        keys, cap, grows = ctx.table_info()
    finally:
        ctx.close()
    plain = sorted(t for i, t in enumerate(submits) if i not in {g["batch"] for g in grows_at})
    return {"batches": len(submits), "initial_capacity": cap0, "final_keys": keys, "final_capacity": cap, "grows": grows,
            "table_mb": round(cap * 1.5 * 16 / 1e6, 1), "median_plain_submit_s": plain[len(plain) // 2] if plain else None,
            "growths": grows_at}


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="directory for the JSON lines")
    ap.add_argument("--records", type=int, default=25_200_000)
    ap.add_argument("--parent", help="source tree of the CLI to compare with (built in place)")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    sys.path.insert(0, ROOT)
    import __graft_entry__
    __graft_entry__.build()
    if args.parent:
        subprocess.run([sys.executable, "-c", "import __graft_entry__ as g; g.build()"], cwd=args.parent, check=True)
    tmp = tempfile.mkdtemp(prefix="uniq_growth_bench_")
    lines = []

    def emit(x):
        print(json.dumps(x), flush=True)
        lines.append(x)
    try:
        src = os.path.join(tmp, "distinct.fa")
        size = write_records(src, args.records)
        dst = os.path.join(tmp, "out.fa")
        r = run_cli(ROOT, src, dst)
        same = r["exit"] == 0 and filecmp.cmp(src, dst, shallow=False)
        emit({"run": "new", "records": args.records, "input_mb": size / 1e6, **r, "output_equals_input": same, **gpu_info()})
        if os.path.exists(dst):
            os.remove(dst)
        if args.parent:
            emit({"run": "parent", "records": args.records, **run_cli(args.parent, src, dst), **gpu_info()})
            if os.path.exists(dst):
                os.remove(dst)
        emit({"run": "growth_trace", **growth_trace(src), **gpu_info()})
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    with open(os.path.join(args.out, "uniq_growth_bench.jsonl"), "w") as f:
        f.write("".join(json.dumps(x) + "\n" for x in lines))
    return 0 if lines and lines[0]["output_equals_input"] else 1


if __name__ == "__main__":
    sys.exit(main())
