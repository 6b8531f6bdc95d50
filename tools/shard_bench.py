"""A run in shard jobs against one run() on the north-star shape (10k segments x 1000 tracks, nucleotide-overlap):
each shard job's time and the share of its histogram pass, the shard files' sizes, the merge's time, the time to
combine all shard files into one (combineShards, where the tree has it), and their sum against one run() of all
samples.  Prints one JSON line.

    python tools/shard_bench.py [--samples 200000] [--shards 4] [--out FILE] [--tree DIR] [--keep DIR]

--tree measures the gat_b200 package of another checkout (with its library built) with this script; --keep leaves
the shard files in DIR.  tools/shard_ab.py alternates two trees this way.

The shard jobs run one after the other in this process (as separate jobs would, each uploads and indexes its inputs
again; the library's pools are warm after a warm-up run of both paths).  The merged statistics are compared with ==
against run()'s.  The card's name and power limit are read in the same call (nvidia-smi query).
"""
import argparse
import hashlib
import json
import os
import shutil
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if "--tree" in sys.argv:
    sys.path.insert(0, os.path.abspath(sys.argv[sys.argv.index("--tree") + 1]))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from tools.hist_bench import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--segments", type=int, default=10000)
    ap.add_argument("--tracks", type=int, default=1000)
    ap.add_argument("--samples", type=int, default=200000)
    ap.add_argument("--shards", type=int, default=4)
    ap.add_argument("--out", default=None)
    ap.add_argument("--tree", default=None)
    ap.add_argument("--keep", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("shard_bench: no CUDA device")

    import gat_b200
    from gat_b200 import engine as Engine, matrixfree, parallel, synthetic
    name, power = card()
    segments, annotations, workspaces, _ = synthetic.make(n_segments=args.segments, n_annotations=args.tracks)
    workspace = synthetic.prepare(segments, annotations, workspaces)
    A = len(list(annotations.tracks))
    counters = [Engine.CounterNucleotideOverlap()]
    tmp = tempfile.mkdtemp(prefix="shard_bench_")
    if args.keep:
        os.makedirs(args.keep, exist_ok=True)

    def timed(fn, *a, **kw):
        Engine.seed(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn(segments, annotations, workspace, Engine.SamplerAnnotator(), counters, Engine.UnconditionalWorkspace(),
                 *a, **kw)
        torch.cuda.synchronize()
        return out, time.perf_counter() - t0

    def table(res):
        return np.array([[r.expected, r.stddev, r.lower95, r.upper95, r.fold, r.pvalue] for r in res])

    try:
        warm = min(args.samples, 20000)                   # module loads, pools
        timed(gat_b200.run, num_samples=warm)
        timed(gat_b200.runShard, (0, warm), os.path.join(tmp, "warm.npz"), num_samples=warm)
        gat_b200.mergeShards([os.path.join(tmp, "warm.npz")])

        whole, run_s = timed(gat_b200.run, num_samples=args.samples)
        jobs, files = [], []
        for k in range(args.shards):
            rng = parallel.shard_range(args.samples, k, args.shards)
            f = os.path.join(args.keep or tmp, "shard%i.npz" % k)
            _, dt = timed(gat_b200.runShard, rng, f, num_samples=args.samples)
            jobs.append({"range": list(rng), "seconds": round(dt, 3),
                         "pass2_seconds": round(matrixfree.info["pass2_seconds"], 3),
                         "pass2_share": round(matrixfree.info["pass2_seconds"] / dt, 4),
                         "resampled": matrixfree.info["reruns"], "arena_bytes": matrixfree.info["arena_bytes"],
                         "file_bytes": os.path.getsize(f)})
            files.append(f)
        t0 = time.perf_counter()
        merged = gat_b200.mergeShards(files)
        merge_s = time.perf_counter() - t0
        identical = bool(np.array_equal(table(whole), table(merged))) and \
            [str(x) for x in whole] == [str(x) for x in merged]
        combine_s = combined_identical = None
        if hasattr(gat_b200, "combineShards"):
            one = os.path.join(tmp, "combined.npz")
            t0 = time.perf_counter()
            gat_b200.combineShards(files, one)
            combine_s = time.perf_counter() - t0
            combined_identical = [str(x) for x in gat_b200.mergeShards([one])] == [str(x) for x in whole]
        digest = hashlib.md5(table(merged).tobytes() + "\n".join(str(x) for x in merged).encode()).hexdigest()
    finally:
        shutil.rmtree(tmp, ignore_errors=True)

    total = sum(j["seconds"] for j in jobs) + merge_s
    report = {"gpu": name, "power_limit": power, "segments": args.segments, "tracks": A,
              "counter": "nucleotide-overlap", "samples": args.samples, "shards": args.shards,
              "run_seconds": round(run_s, 3), "shard_jobs": jobs, "merge_seconds": round(merge_s, 3),
              "shard_files_bytes": sum(j["file_bytes"] for j in jobs),
              "shards_plus_merge_seconds": round(total, 3), "over_one_run": round(total / run_s, 3),
              "statistics_identical": identical, "combine_seconds": None if combine_s is None else round(combine_s, 3),
              "combined_identical": combined_identical, "statistics_md5": digest,
              "package": os.path.dirname(gat_b200.__file__)}
    line = json.dumps(report)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
