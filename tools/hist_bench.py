"""Matrix mode against matrix-free mode of gat_b200.run() (keep_samples=True / False) on the north-star shape,
and one run whose sample matrix cannot fit in GPU memory.  Prints one JSON line.

    python tools/hist_bench.py [--samples 200000] [--reps 3] [--big-samples 60000000] [--out FILE]

- samples/s of run() in both modes, alternating in one process (the problem and the seed are the same; the
  statistics of the two modes are compared with ==);
- device ms per slab of the two kernels the matrix-free mode adds (CUDA events over repeated launches on one
  slab of real counts): the accumulating pass 1 and the quantile-window histogram;
- --big-samples: run() with the default keep_samples=None at a size whose matrix exceeds the free memory (the
  default picks the matrix-free mode), to completion: wall time and the device memory the run added to what the
  process already held from the runs before it (the largest drop of free memory, cudaMemGetInfo, seen after each
  slab; the annotation index and batch buffers are pooled by then).
The card's name and power limit are read in the same call (nvidia-smi query).
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power = (q.stdout.strip().split(", ") + ["?", "?"])[:2]
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--segments", type=int, default=10000)
    ap.add_argument("--tracks", type=int, default=1000)
    ap.add_argument("--samples", type=int, default=200000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--big-samples", type=int, default=60000000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("hist_bench: no CUDA device")

    import gat_b200
    from gat_b200 import device, engine as Engine, matrixfree, synthetic
    name, power = card()
    segments, annotations, workspaces, _ = synthetic.make(n_segments=args.segments, n_annotations=args.tracks)
    workspace = synthetic.prepare(segments, annotations, workspaces)
    A = len(list(annotations.tracks))
    counters = [Engine.CounterNucleotideOverlap()]

    def run(S, keep):
        Engine.seed(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = gat_b200.run(segments, annotations, workspace, Engine.SamplerAnnotator(), counters,
                           Engine.UnconditionalWorkspace(), num_samples=S, keep_samples=keep)
        torch.cuda.synchronize()
        return res, time.perf_counter() - t0

    def table(res):
        return np.array([[r.expected, r.stddev, r.lower95, r.upper95, r.fold, r.pvalue] for r in res])

    run(min(args.samples, 20000), True)                  # warm-up of both modes (module loads, pools)
    run(min(args.samples, 20000), False)
    rate = {True: [], False: []}
    identical = True
    for _ in range(args.reps):
        got = {}
        for keep in (True, False):
            res, dt = run(args.samples, keep)
            rate[keep].append(args.samples / dt)
            got[keep] = table(res)
        identical = identical and bool(np.array_equal(got[True], got[False]))
    info = dict(matrixfree.info)

    # the two added kernels on one slab of real counts (the slab run() uses: SLAB_BYTES / (4 A) rows)
    ctx = Engine.getContext()
    rows = info["chunk_rows"]
    smp, annos = gat_b200.trackSampler(segments[list(segments.tracks)[0]], annotations, workspace, Engine.SamplerAnnotator())
    slab = torch.zeros(rows * A, dtype=torch.int32, device="cuda")
    ctx.set_stream(torch.cuda.current_stream().cuda_stream or 1)
    smp.run(annos, ["nucleotide-overlap"], 1, 0, 0, rows, out_counts_ptr=slab.data_ptr())
    st = ctx.column_stats(None, np.zeros(A), device_ptr=slab.data_ptr(), n_samples=rows, n_cols=A, is_float=0)
    lo, hi = matrixfree.pilot_windows(st["lower95"], st["upper95"])
    acc = device.ColumnAccumulator(ctx, A, 1 << 31, np.zeros(A))
    acc.set_windows(lo.astype(np.uint32), (hi - lo + 1).astype(np.uint32))
    kernel_ms = {}
    for what, kw in (("pass1_sums", dict(sums=True, hist=False)), ("window_histogram", dict(sums=False, hist=True))):
        for _ in range(3):
            acc.add(slab.data_ptr(), rows, A, **kw)
        n = 20
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            acc.add(slab.data_ptr(), rows, A, **kw)
        e1.record()
        torch.cuda.synchronize()
        kernel_ms[what] = e0.elapsed_time(e1) / n
    acc.close()
    smp.close()
    annos.close()
    ctx.set_stream(None)

    report = {"gpu": name, "power_limit": power, "segments": args.segments, "tracks": A, "counter": "nucleotide-overlap",
              "samples": args.samples, "reps": args.reps,
              "matrix_samples_per_s": round(float(np.median(rate[True])), 1),
              "matrix_free_samples_per_s": round(float(np.median(rate[False])), 1),
              "matrix_free_over_matrix": round(float(np.median(rate[False]) / np.median(rate[True])), 4),
              "statistics_identical": identical, "slab_rows": rows, "slab_bytes": 4 * rows * A,
              "arena_bytes": info["arena_bytes"], "reruns": info["reruns"],
              "kernel_ms_per_slab": dict((k, round(v, 4)) for k, v in kernel_ms.items()),
              "slab_gb_per_s": dict((k, round(4 * rows * A / (v * 1e-3) / 1e9, 1)) for k, v in kernel_ms.items())}

    if args.big_samples:
        S = args.big_samples
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        peak, slabs = [0], [0]
        orig = matrixfree.stream_statistics

        def spy(ctx, produce, *a, **kw):
            def produce_and_measure(r0, n):
                ptr = produce(r0, n)
                slabs[0] += 1
                torch.cuda.synchronize()
                peak[0] = max(peak[0], free0 - torch.cuda.mem_get_info()[0])
                return ptr
            return orig(ctx, produce_and_measure, *a, **kw)
        matrixfree.stream_statistics = spy
        try:
            res, dt = run(S, None)
        finally:
            matrixfree.stream_statistics = orig
        report["big"] = {"samples": S, "matrix_bytes": 4 * S * A, "free_bytes_before": free0,
                         "matrix_free_slabs": slabs[0], "seconds": round(dt, 2), "samples_per_s": round(S / dt, 1),
                         "device_bytes_added": peak[0], "arena_bytes": matrixfree.info["arena_bytes"],
                         "reruns": matrixfree.info["reruns"], "results": len(res),
                         "nsamples": res[0].nsamples if res else 0}
    line = json.dumps(report)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
