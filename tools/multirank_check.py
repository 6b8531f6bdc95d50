"""N-rank identity check of gat_b200.run over NCCL (VERDICT r1, weak #1d): the matrix and the statistics an N-rank
run produces must equal the 1-rank run's, for both exchange routes (all-gather of the sample slabs, all-to-all by
column) and a number of samples that N does not divide.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        tools/multirank_check.py [--samples 10007] [--tracks 40] [--keep-samples 0]

--keep-samples 0: the sharded run is the matrix-free mode (run(..., keep_samples=False)), against the 1-rank
matrix run.

Every rank first runs the problem alone (no process group: world = 1), then joins the group and runs it sharded;
rank 0 prints one JSON line.  Exit code 1 on any difference.
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=10007)
    ap.add_argument("--tracks", type=int, default=40)
    ap.add_argument("--segments", type=int, default=10000)
    ap.add_argument("--isochores", action="store_true")
    ap.add_argument("--keep-samples", type=int, default=1)
    args = ap.parse_args()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)

    import gat_b200
    from gat_b200 import engine as Engine, parallel, synthetic

    # (integer counters: the peer transport routes them; a density counter makes run() use NCCL for everything)
    names = ["nucleotide-overlap", "segment-overlap", "annotation-overlap"]

    def run(**kw):
        segments, annotations, workspaces, iso = synthetic.make(args.segments, args.tracks, 5000, isochores=args.isochores)
        workspace = synthetic.prepare(segments, annotations, workspaces, iso)
        Engine.seed(7)
        t0 = time.perf_counter()
        res = gat_b200.run(segments, annotations, workspace, Engine.SamplerAnnotator(),
                           [Engine.COUNTER_CLASSES[n]() for n in names], Engine.UnconditionalWorkspace(),
                           num_samples=args.samples, **kw)
        torch.cuda.synchronize()
        return res, time.perf_counter() - t0

    def table(res):
        return np.array([[r.observed, r.expected, r.stddev, r.lower95, r.upper95, r.fold, r.pvalue] for r in res])

    alone, t_alone = run()                              # world = 1: the reference matrix
    assert parallel.init_from_env(), "launch with torch.distributed.run"
    rank, world = parallel.rank_world()
    report = {"ranks": world, "samples": args.samples, "tracks": args.tracks, "counters": names,
              "isochores": args.isochores, "seconds_1_rank": round(t_alone, 3)}
    ok = True
    modes = (("allgather", dict(exchange="allgather", transport="nccl")),
             ("columns", dict(exchange="columns", transport="nccl")),
             ("peer_allgather", dict(exchange="allgather", transport="peer")),
             ("peer_columns", dict(exchange="columns", transport="peer")))
    if not args.keep_samples:
        modes = (("matrix_free", dict(keep_samples=False)),)
    for mode, kw in modes:
        got, dt = run(**kw)
        same_stats = bool(np.array_equal(table(alone), table(got)))
        n_cols = n_equal = 0
        for a, g in zip(alone, got):
            assert (a.track, a.annotation, a.counter) == (g.track, g.annotation, g.counter)
            try:
                mine = g.samples
            except RuntimeError:                        # column-sharded: the column lives on another rank (or
                continue                                # the samples were not kept)
            n_cols += 1
            n_equal += int(np.array_equal(a.samples, mine))
        flags = torch.tensor([int(same_stats), n_cols, n_equal], dtype=torch.int64, device="cuda")
        torch.distributed.all_reduce(flags)
        report[mode] = {"statistics_equal_on_ranks": int(flags[0]), "sample_columns_checked": int(flags[1]),
                        "sample_columns_equal": int(flags[2]), "seconds": round(dt, 3)}
        expect_cols = 0 if mode == "matrix_free" else len(alone) * (world if mode.endswith("allgather") else 1)
        ok = ok and int(flags[0]) == world and int(flags[1]) == int(flags[2]) == expect_cols
    report["ok"] = ok
    if rank == 0:
        print(json.dumps(report))
    parallel.finalize()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
