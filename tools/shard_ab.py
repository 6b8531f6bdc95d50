"""tools/shard_bench.py on two checkouts, alternated in fresh processes, with the medians of each: shard job time and
its pass-2 share, merge time, combine time (where a tree has combineShards), whether the statistics equal run()'s
and each other's, and whether the two trees wrote the same shard file arrays.  Prints one JSON line.

    python tools/shard_ab.py --trees PARENT_DIR . [--rounds 3] [--samples 200000] [--shards 4] [--out FILE]

Each tree needs its library built (make -C gat_b200/csrc).
"""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def same_files(a, b):
    """the shard files of two trees hold the same arrays (names, dtypes, values)"""
    for name in sorted(os.listdir(a)):
        with np.load(os.path.join(a, name)) as x, np.load(os.path.join(b, name)) as y:
            if sorted(x.files) != sorted(y.files):
                return False
            for k in x.files:
                if x[k].dtype != y[k].dtype or x[k].shape != y[k].shape or \
                        not np.array_equal(x[k], y[k], equal_nan=x[k].dtype.kind == "f"):   # (no reference: NaN folds)
                    return False
    return True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--trees", nargs=2, required=True)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--samples", type=int, default=200000)
    ap.add_argument("--shards", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    runs = dict((t, []) for t in args.trees)
    tmp = tempfile.mkdtemp(prefix="shard_ab_")
    try:
        for r in range(args.rounds):
            for t in (args.trees if r % 2 == 0 else args.trees[::-1]):
                keep = os.path.join(tmp, "tree%i" % args.trees.index(t))
                shutil.rmtree(keep, ignore_errors=True)
                out = subprocess.run([sys.executable, os.path.join(HERE, "shard_bench.py"), "--tree", t, "--keep", keep,
                                      "--samples", str(args.samples), "--shards", str(args.shards)],
                                     capture_output=True, text=True, check=True)
                runs[t].append(json.loads(out.stdout.strip().splitlines()[-1]))
        files_identical = same_files(os.path.join(tmp, "tree0"), os.path.join(tmp, "tree1"))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)

    def med(xs):
        xs = [x for x in xs if x is not None]
        return round(statistics.median(xs), 3) if xs else None
    report = {"gpu": runs[args.trees[0]][0]["gpu"], "power_limit": runs[args.trees[0]][0]["power_limit"],
              "samples": args.samples, "shards": args.shards, "rounds": args.rounds, "trees": {}}
    for t, rs in runs.items():
        jobs = [j for r in rs for j in r["shard_jobs"]]
        report["trees"][t] = {
            "run_seconds": med([r["run_seconds"] for r in rs]),
            "shard_job_seconds": med([j["seconds"] for j in jobs]),
            "pass2_seconds": med([j["pass2_seconds"] for j in jobs]), "pass2_share": med([j["pass2_share"] for j in jobs]),
            "merge_seconds": med([r["merge_seconds"] for r in rs]),
            "combine_seconds": med([r["combine_seconds"] for r in rs]),
            "shards_plus_merge_seconds": med([r["shards_plus_merge_seconds"] for r in rs]),
            "over_one_run": med([r["over_one_run"] for r in rs]),
            "shard_files_bytes": rs[0]["shard_files_bytes"],
            "statistics_identical": all(r["statistics_identical"] for r in rs),
            "combined_identical": [r["combined_identical"] for r in rs][0],
            "statistics_md5": sorted(set(r["statistics_md5"] for r in rs))}
    md5 = [v["statistics_md5"] for v in report["trees"].values()]
    report["statistics_equal_across_trees"] = md5[0] == md5[1] and len(md5[0]) == 1
    report["shard_files_equal_across_trees"] = files_identical
    line = json.dumps(report)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
