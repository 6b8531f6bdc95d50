"""A/B timing of placement-kernel builds: several built trees of this repository, alternated within each round, one
fresh `bench.py` process per line, and their dumped outputs compared

    python tools/place_ab.py --tree parent=DIR --tree new=DIR [--tree ...] [--configs ns,c2,c3] [--rounds 3]
                             [--out FILE.json]

Each DIR is a copy of the repository with its library already built (`__graft_entry__.build()`).  Per round and
config every tree runs `bench.py --gpus 1 --no-cpu-baseline --no-e2e --config CFG` from its own directory; the
JSON gives `value` (samples/s), `roofline.other_kernels.place_kernel_ms` and `roofline.kernel_ms` (counting).  Then
every tree runs `bench.py --steps 3 --warmup 1 --dump-outputs` once per config and its `counts.npy` /
`sample_index.npy` are compared with the first tree's.  The GPU's name, power limit and maximum SM clock are read
(nvidia-smi query only) in the same call, since the times belong to them.  Output: medians and spreads (max - min)
per (config, tree) and every line.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

import numpy as np


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.TimeoutExpired):
        return "unknown"


def bench_line(tree, args):
    r = subprocess.run([sys.executable, os.path.join(tree, "bench.py")] + args, cwd=tree, capture_output=True,
                       text=True)
    if r.returncode != 0:
        raise RuntimeError("bench.py in %s failed (%d):\n%s" % (tree, r.returncode, r.stderr[-3000:]))
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    return json.loads(lines[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tree", action="append", required=True, help="NAME=DIR")
    ap.add_argument("--configs", default="ns,c2,c3")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    trees = [(name, os.path.abspath(d)) for name, d in (t.split("=", 1) for t in args.tree)]
    configs = args.configs.split(",")
    result = {"gpu": gpu_info(),
              "command": "python bench.py --gpus 1 --no-cpu-baseline --no-e2e --config CFG (trees alternated within "
                         "each round, one fresh process per line, %d rounds)" % args.rounds,
              "trees": [name for name, _ in trees], "runs": []}
    for rnd in range(1, args.rounds + 1):
        for cfg in configs:
            for name, tree in trees:
                d = bench_line(tree, ["--gpus", "1", "--no-cpu-baseline", "--no-e2e", "--config", cfg])
                run = {"tree": name, "round": rnd, "config": cfg, "value": d["value"],
                       "place_kernel_ms": d["roofline"]["other_kernels"]["place_kernel_ms"],
                       "count_kernel_ms": d["roofline"]["kernel_ms"], "parity_check": d["parity_check"]}
                result["runs"].append(run)
                print(json.dumps(run), flush=True)
    summary = {}
    for cfg in configs:
        for name, _ in trees:
            rs = [r for r in result["runs"] if r["tree"] == name and r["config"] == cfg]
            v = [r["value"] for r in rs]
            p = [r["place_kernel_ms"] for r in rs]
            summary["%s/%s" % (cfg, name)] = {
                "value_median": round(statistics.median(v)), "value_spread": round(max(v) - min(v)),
                "place_kernel_ms_median": round(statistics.median(p), 4),
                "place_kernel_ms_spread": round(max(p) - min(p), 4), "n": len(rs)}
    result["summary"] = summary
    outputs = {}
    with tempfile.TemporaryDirectory() as tmp:
        for cfg in configs:
            ref = None
            for name, tree in trees:
                d = os.path.join(tmp, "%s_%s" % (cfg, name))
                bench_line(tree, ["--gpus", "1", "--no-cpu-baseline", "--no-e2e", "--config", cfg, "--steps", "3",
                                  "--warmup", "1", "--dump-outputs", d])
                arrs = [np.load(os.path.join(d, f)) for f in ("counts.npy", "sample_index.npy")]
                if ref is None:
                    ref = arrs
                    outputs["%s/%s" % (cfg, name)] = "reference (counts %s)" % (arrs[0].shape,)
                else:
                    same = all(np.array_equal(a, b) for a, b in zip(arrs, ref))
                    outputs["%s/%s" % (cfg, name)] = "identical" if same else "DIFFERENT"
    result["outputs"] = outputs
    print(json.dumps({"summary": summary, "outputs": outputs, "gpu": result["gpu"]}, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
