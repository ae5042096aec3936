"""End-to-end measurement of `python -m circkit_b200 monomerize` (or canonicalize / uniq) on a FASTA file (one GPU).

    python tools/mono_stream_bench.py --out DIR [--command canonicalize|uniq|monomerize] [--parent TREE] [--records 1000000]
                                      [--scale 4]

Writes data of bench.py's `--workload mono` shape (1 M concatemers: 2.3 copies of a 250-400 nt unit, 1 % substitutions;
bench.py's unit lengths and base hash, generated on the device in blocks) as FASTA with 70-column lines to a temporary
directory, runs the CLI's --command on it (monomerize, the default: with seed 10 and min identity 0.95), and prints one JSON line per run: wall time, records/s, input MB/s and the child's peak RSS, with the card's name and
power limit read in the same process.  --parent TREE: the CLI of another source tree (e.g. an exported copy of an earlier
commit, built in place) runs on the same file and the two outputs are compared byte for byte.  --scale K: a second file K
times as large goes through this tree's CLI only, to show whether peak RSS grows with the input.
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

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.splitlines()[0].split(", ") + ["?"])[:2] if q.returncode == 0 and q.stdout else ("?", "?")
    return {"gpu": name.strip(), "power_limit": power.strip()}


def write_fasta(path: str, n: int, seed_offset: int = 0) -> int:
    """bench.py's mono workload (its generator, record ids offset by seed_offset), 70-column lines; returns the file size"""
    import numpy as np
    import torch
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(1 + seed_offset)
    unit_len = rng.integers(250, 401, n)
    total_len = (unit_len * 2.3).astype(np.int64)
    off = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(total_len, out=off[1:])
    with open(path, "wb") as f:
        block = 250_000
        g = torch.Generator(device=dev).manual_seed(7 + seed_offset)
        letters = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device=dev)
        for lo in range(0, n, block):
            hi = min(n, lo + block)
            tl = torch.from_numpy(total_len[lo:hi]).to(dev)
            o = torch.from_numpy(off[lo:hi + 1] - off[lo]).to(dev)
            rec = torch.repeat_interleave(torch.arange(lo, hi, device=dev), tl)
            pos = torch.arange(int(o[-1]), device=dev) - o[rec - lo]
            h = (rec * 1000003 + (pos % torch.from_numpy(unit_len[lo:hi]).to(dev)[rec - lo])) * 2654435761 % 4294967296
            raw = letters[((h >> 13) ^ (h >> 7)) & 3]
            mut = torch.rand(raw.numel(), device=dev, generator=g) < 0.01
            raw[mut] = letters[torch.randint(0, 4, (int(mut.sum()),), device=dev, generator=g)]
            arena = raw.cpu().numpy().tobytes()
            oo = (off[lo:hi + 1] - off[lo]).tolist()
            parts = []
            for i in range(hi - lo):
                s = arena[oo[i]: oo[i + 1]]
                parts.append(b">m%d\n" % (lo + i) + b"\n".join(s[k: k + 70] for k in range(0, len(s), 70)) + b"\n")
            f.write(b"".join(parts))
    torch.cuda.empty_cache()
    return os.path.getsize(path)


def run_cli(tree: str, command: str, src: str, dst: str) -> dict:
    """one `python -m circkit_b200 COMMAND` child in `tree`: wall time and peak RSS (its own rusage, from wait4)"""
    cmd = [sys.executable, "-m", "circkit_b200", command, src, "-o", dst]
    if command == "monomerize":
        cmd += ["--seed-length", "10", "--min-identity", "0.95"]
    env = dict(os.environ, PYTHONPATH=tree)
    t0 = time.perf_counter()
    p = subprocess.Popen(cmd, cwd=tree, env=env)
    _, status, ru = os.wait4(p.pid, 0)
    wall = time.perf_counter() - t0
    p.returncode = os.waitstatus_to_exitcode(status)
    return {"exit": p.returncode, "wall_s": wall, "peak_rss_mb": ru.ru_maxrss / 1024}


def report(label: str, tree: str, command: str, src: str, n: int, size: int, dst: str) -> dict:
    r = run_cli(tree, command, src, dst)
    line = {"run": label, "command": command, "tree": os.path.basename(os.path.abspath(tree)), "records": n, "input_mb": size / 1e6, **r,
            "records_per_s": n / r["wall_s"], "input_mb_per_s": size / 1e6 / r["wall_s"], **gpu_info()}
    print(json.dumps(line), flush=True)
    return line


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="directory for the JSON lines")
    ap.add_argument("--command", choices=["canonicalize", "uniq", "monomerize"], default="monomerize")
    ap.add_argument("--parent", help="source tree of the CLI to compare with (built in place)")
    ap.add_argument("--records", type=int, default=1_000_000)
    ap.add_argument("--scale", type=int, default=4)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    sys.path.insert(0, ROOT)
    import __graft_entry__
    __graft_entry__.build()
    if args.parent:
        subprocess.run([sys.executable, "-c", "import __graft_entry__ as g; g.build()"], cwd=args.parent, check=True)
    tmp = tempfile.mkdtemp(prefix="mono_stream_bench_")
    try:
        src = os.path.join(tmp, "mono_1x.fa")
        size = write_fasta(src, args.records)
        lines = [report("new", ROOT, args.command, src, args.records, size, os.path.join(tmp, "new_1x.fa"))]
        if args.parent:
            lines.append(report("parent", args.parent, args.command, src, args.records, size, os.path.join(tmp, "parent_1x.fa")))
            same = filecmp.cmp(os.path.join(tmp, "new_1x.fa"), os.path.join(tmp, "parent_1x.fa"), shallow=False)
            print(json.dumps({"outputs_identical": same}), flush=True)
            lines.append({"outputs_identical": same})
        for f in os.listdir(tmp):
            os.remove(os.path.join(tmp, f))
        if args.scale > 1:
            big = os.path.join(tmp, "mono_%dx.fa" % args.scale)
            bsize = write_fasta(big, args.records * args.scale)
            lines.append(report("new_%dx" % args.scale, ROOT, args.command, big, args.records * args.scale, bsize,
                                os.path.join(tmp, "new_%dx.fa" % args.scale)))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    name = "mono_stream_bench.jsonl" if args.command == "monomerize" else "mono_stream_bench_%s.jsonl" % args.command
    with open(os.path.join(args.out, name), "w") as f:
        f.write("".join(json.dumps(x) + "\n" for x in lines))
    return 0 if all(x.get("exit", 0) == 0 for x in lines) and all(x.get("outputs_identical", True) for x in lines) else 1


if __name__ == "__main__":
    sys.exit(main())
