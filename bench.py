#!/usr/bin/env python
"""bench.py -- samples/sec of the GAT simulation hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config ns|c2|c3|c4|c5]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

Workload (config.workload): by default the metric's own shape ("ns") -- synthetic hg19 (24 contigs), 10 000
segments against 1 000 annotation tracks of 20 000 intervals, contig workspace, nucleotide-overlap counter;
--config c2..c5 are the other BASELINE.json configurations (50 tracks; 8 GC isochores + segment-overlap;
50 000 segments x 1 000 tracks; 200 tracks).
A step = one pass of the hot path (placement of every unit + counting against every annotation) over
`--batches-per-step` internal batches of `--batch` Monte-Carlo samples per GPU (default 24 x 4096 = 98 304 samples,
~60 ms on one B200, so that 20 steps are > 1 s of sustained load); sample indices advance every step, so no step
repeats another's work.  Weak scaling: every rank runs the same number of samples on its own shard of the global
sample index space; for N > 1 the per-step count slab is all-gathered over NCCL (the path's one exchange step)
inside the timed region; the all-gather of a step runs asynchronously and overlaps the next step's kernels (two
output slabs), the last ones are waited for before the closing event.

value   whole-job samples/s, inputs resident in HBM, counts left in HBM (CUDA events, max over ranks)
e2e     same metric through the C ABI with HOST buffers: every step uploads segments, workspace and annotations
        from pinned host memory (gatb_sampler_create / gatb_annotations_create_async), runs, (N > 1: all-gathers
        the slab,) and reads the step's count matrix back to pinned host memory; double-buffered -- the annotation
        upload and index build of step i+1 are queued before gatb_run of step i and overlap its kernels
parity_check   two samples of the last timed step's slab recomputed by the CPU oracle (outside the timed region)
gather_check   N > 1: every rank's rows of the gathered matrix of one step recomputed on rank 0 alone
roofline  dominant kernel (counting), see roofline_of(): output-sensitive bytes against the measured L2 peak,
          compulsory DRAM bytes against the measured HBM peak, issue rate against the measured issue peak
cpu_baseline  the reference itself (oracle/_ref) on the host cores, bounded sample, rank 0, N=1
"""
import argparse
import collections
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

UNIT = "samples/s"
SEED = 20260101
DUMP_BYTES = 32 << 20          # --dump-outputs: rows of the count matrix kept

# BASELINE.json configs: (segments, annotation tracks, isochores, counter, metric label)
CONFIGS = {
    "ns": dict(segments=10000, annotations=1000, isochores=False, counter="nucleotide-overlap",
               metric="samples/sec (10k segs x 1k annotations)"),
    "c2": dict(segments=10000, annotations=50, isochores=False, counter="nucleotide-overlap",
               metric="samples/sec (10k segs x 50 annotations)"),
    "c3": dict(segments=10000, annotations=50, isochores=True, counter="segment-overlap",
               metric="samples/sec (10k segs x 50 annotations, 8 GC isochores, segment-overlap)"),
    "c4": dict(segments=50000, annotations=1000, isochores=False, counter="nucleotide-overlap",
               metric="samples/sec (50k segs x 1k annotations)"),
    "c5": dict(segments=10000, annotations=200, isochores=False, counter="nucleotide-overlap",
               metric="samples/sec (10k segs x 200 annotations)"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="ns", choices=sorted(CONFIGS))
    ap.add_argument("--segments", type=int, default=None)
    ap.add_argument("--annotations", type=int, default=None)
    ap.add_argument("--annotation-intervals", type=int, default=20000)
    ap.add_argument("--batch", type=int, default=4096, help="samples per internal placement / counting batch")
    ap.add_argument("--batches-per-step", type=int, default=24)
    ap.add_argument("--counter", default=None)
    ap.add_argument("--isochores", action="store_true", default=None)
    ap.add_argument("--cpu-samples", type=int, default=0, help="reference samples (0 = about 10-30 s worth)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-checks", action="store_true")
    ap.add_argument("--e2e-device-path", action="store_true",
                    help="diagnostic: at N = 1 run the e2e leg the way N > 1 does (device output, side-stream read-back)")
    ap.add_argument("--gather", default="peer", choices=["peer", "peer-kernel", "nccl"],
                    help="N > 1: how the per-step count slabs reach every rank -- peer: output routes into every rank's "
                         "matrix over NVLink, served by copy engines behind the next batch; peer-kernel: the same routes "
                         "served by the counting kernel's own stores; nccl: all_gather_into_tensor")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a fixed, seeded sample of rows of the last timed step's count "
                         "matrix (DIR/counts.npy, float64) and their global sample indices (DIR/sample_index.npy)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    cfg = CONFIGS[args.config]
    for k in ("segments", "annotations", "counter", "isochores"):
        if getattr(args, k) is None:
            setattr(args, k, cfg[k])
    args.metric = cfg["metric"]
    args.samples_per_step = args.batch * args.batches_per_step
    return args


# ------------------------------------------------------------------------------------------- workload
def build_workload(args):
    """synthetic inputs, prepared as gat-run.py prepares them, flattened to the CSR of the C ABI"""
    import gat_b200
    from gat_b200 import synthetic, device
    segments, annotations, workspaces, iso = synthetic.make(args.segments, args.annotations,
                                                            args.annotation_intervals, isochores=args.isochores)
    workspace = synthetic.prepare(segments, annotations, workspaces, iso)
    problem = gat_b200.TrackProblem(segments["merged"], workspace)
    atracks, lists, nseg = gat_b200.buildContigAnnotations(annotations, workspace, problem.contigs)
    A, C = len(atracks), len(problem.contigs)
    anno_csr = device.to_csr([lists[a][c] for a in range(A) for c in range(C)])
    seg_csr = device.to_csr(problem.unit_segments)
    ws_csr = device.to_csr(problem.unit_workspace)
    n_a_total = int(anno_csr[0][-1])
    wl = dict(problem=problem, A=A, C=C, nseg=np.array(nseg, dtype=np.uint32), anno_csr=anno_csr, seg_csr=seg_csr,
              ws_csr=ws_csr, n_a_total=n_a_total, n_segments=int(seg_csr[0][-1]), lists=lists,
              collections=(segments, annotations, workspace))
    return wl


def config_of(args, wl, world):
    return {"workload": "%s: synthetic hg19 (24 contigs, contig workspace%s): %i segments x %i annotation tracks "
                        "(%i intervals after normalize), counter %s, sampler annotator"
                        % (args.config, ", 8 GC isochores" if args.isochores else "", wl["n_segments"], wl["A"],
                           wl["n_a_total"], args.counter),
            "samples_per_step_per_gpu": args.samples_per_step,
            "batch": args.batch, "batches_per_step": args.batches_per_step,
            "global_samples_per_step": args.samples_per_step * world,
            "parallelism": ("samples sharded over %i GPU(s), inputs replicated; exchange per step: %s" % (world, (
                "output routes (gatb_set_output_routes) into every rank's [N x samples][tracks] matrix in CUDA IPC peer "
                "memory over NVLink -- no collective; served by " + ("the counting kernel's own stores" if
                args.gather == "peer-kernel" else "copy engines while the next batch runs") if args.gather != "nccl" else
                "one NCCL all_gather_into_tensor of the count slab, overlapping the next step's kernels"))) if world > 1 else "1 GPU",
            "l2": "inputs larger than L2: annotation grid index ~%.0f MB + %.0f MB of placed segments per batch; "
                  "sample indices advance every step"
                  % (wl["n_a_total"] * 2.33 * 8 / 1e6 + 12, args.batch * wl["n_segments"] * 8 / 1e6),
            "data_seed": SEED}


def dump_outputs(directory, matrix, sample_index):
    """the count matrix of a step as a caller of the path receives it ([samples][annotation tracks] on the device),
    reduced to whole rows picked by a generator with a fixed seed, so that two builds run with the same arguments
    can be compared output for output; at most DUMP_BYTES of float64 (exact for uint32 counts)"""
    import torch
    os.makedirs(directory, exist_ok=True)
    rows, cols = matrix.shape
    n = min(rows, max(1, DUMP_BYTES // (8 * cols)))
    pick = np.sort(np.random.default_rng(SEED).choice(rows, n, replace=False))
    if matrix.dtype == torch.uint32:
        matrix = matrix.view(torch.int32)
    sample = matrix.index_select(0, torch.from_numpy(pick).to(matrix.device)).cpu().numpy()
    if sample.dtype == np.int32:
        sample = sample.view(np.uint32)
    np.save(os.path.join(directory, "counts.npy"), sample.astype(np.float64))
    np.save(os.path.join(directory, "sample_index.npy"), np.asarray(sample_index)[pick].astype(np.float64))


# --------------------------------------------------------------------------------------------- clocks
class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons while the timed region runs"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def mark(self):
        return time.perf_counter()

    def stop(self, t_begin=None, t_end=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, row in self.rows:
            if t_begin is not None and not (t_begin <= t <= t_end):
                continue
            f = [x.strip() for x in row.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(power) if power else None}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_facts():
    """per-launch facts of the counting kernel that only ncu can give (warp instructions, DRAM bytes), from the
    committed capture of the same command (profiles/count_kernel_traffic.json)"""
    p = os.path.join(ROOT, "profiles", "count_kernel_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


def microbench(lib, device_index):
    out = {}
    buf = np.zeros(4, dtype=np.float64)
    from gat_b200 import device
    if lib.gatb_microbench(device_index, 0, 48 << 20, 5, device._p(buf)) == 0:
        out["l2_read_gbs"] = float(buf[0])
    if lib.gatb_microbench(device_index, 1, 0, 5, device._p(buf)) == 0:
        out["issue_gwarp_inst_s"] = float(buf[0])
        out["sms"] = int(buf[3])
    return out


# ---------------------------------------------------------------------------------------- reference arm
def reference_rate(args, wl, seconds_target=15.0):
    """the reference's UnconditionalSampler.sample on this box's host cores: single process and its
    multiprocessing path, each on a bounded sample; returns the faster with both reported"""
    from oracle import ref_bench
    segments, annotations, workspace = wl["collections"]
    cores = os.cpu_count() or 1
    # probe to size the sample
    dt, _ = ref_bench.time_sampling(segments, annotations, workspace, [args.counter], 2, num_threads=0)
    per = dt / 2
    n1 = args.cpu_samples or int(max(4, min(200, seconds_target / max(per, 1e-3))))
    dt1, _ = ref_bench.time_sampling(segments, annotations, workspace, [args.counter], n1, num_threads=0)
    r1 = n1 / dt1
    # its multiprocessing path (--num-threads): the parent re-pickles ALL interval arrays for every task
    # (SURVEY section 5), so throughput stops growing after a few workers; at most 32 workers, one
    # sample per worker, keeps this leg bounded on many-core hosts
    workers = min(cores, 32)
    nm = workers
    rm, dtm = None, None
    try:
        dtm, _ = ref_bench.time_sampling(segments, annotations, workspace, [args.counter], nm, num_threads=workers)
        rm = nm / dtm
    except Exception as e:  # pragma: no cover
        rm = None
        sys.stderr.write("reference multiprocessing path failed: %s\n" % e)
    best, used = (r1, 1)
    if rm is not None and rm > r1:
        best, used = rm, workers
    cores = workers
    sample = ("reference UnconditionalSampler.sample: %i samples single-process in %.1f s (%.3f samples/s); "
              "%s; faster mode reported" %
              (n1, dt1, r1, ("%i samples with --num-threads=%i in %.1f s (%.3f samples/s)" % (nm, cores, dtm, rm))
               if rm is not None else "multiprocessing path failed"))
    return best, used, sample


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref_bench
    if not ref_bench.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref not built (python oracle/build_ref.py)"}))
        return
    wl = build_workload(args)
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    t0 = time.perf_counter()
    rate, cores, sample = reference_rate(args, wl, seconds_target=min(30.0, 20.0 * max(args.steps, 1) / 5.0))
    line = {"metric": args.metric, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 * args.samples_per_step / rate,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32",
            "data": "synthetic", "impl": "reference", "config": config_of(args, wl, world),
            "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample},
            "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------- roofline
def roofline_of(args, wl, ctx, smp, annos, prof, local, sm_mhz=None):
    """The counting kernel against three measured machine limits.  All byte counts are PER LAUNCH (= one batch)
    and recomputable from `config` plus the counters in `work`:

    l2    output-sensitive bytes = 8 * pairs + 8 * P * batch + index_bytes, where pairs = truly overlapping
          (segment, interval) pairs of the batch (sum of the GATB_OVERLAP_PIECES plane: every pair's 8-byte
          index entry has to reach an SM at least once), P = placed segments per sample (8 bytes each, read
          once), index_bytes = offsets + entries of the grid index (read once);  peak = L2 read bandwidth
          measured by gatb_microbench on this GPU.  This is the `roofline` the line reports (frac <= 1).
    hbm   compulsory DRAM bytes = index_bytes + 8 * P * batch + 4 * A * batch (counts out) against the measured
          HBM copy bandwidth (MEASURED_PEAKS.json): how far from HBM-bound the kernel is.
    issue warp instructions per launch (ncu capture of the same command, committed) / kernel time against the
          measured issue peak: what actually limits the kernel.
    reference_algorithm_equivalent: the SURVEY 8d bytes of the reference's two-pointer merge (every cell streams
          its sample and its annotation list) -- what the same answers would cost without the index."""
    from gat_b200 import device
    import torch
    B, A = args.batch, wl["A"]
    count_ms = prof["count"][0] / max(prof["count"][1], 1)
    place_ms = prof["place"][0] / max(prof["place"][1], 1)
    merge_ms = prof["merge"][0] / max(prof["merge"][1], 1)
    # work counters of one batch: pairs from the overlap-pieces counter, tested entries from the index geometry
    dev = torch.device("cuda", local)
    plane = torch.zeros((1, B, A), dtype=torch.int32, device=dev)
    begin = 4 * 10 ** 9            # (its own corner of the sample index space, < 2^32)
    info = smp.run(annos, ["overlap-pieces"], SEED, 0, begin, B, out_counts_ptr=plane.data_ptr())
    pairs = int(plane.to(torch.int64).sum().item())
    work = np.zeros(4, dtype=np.uint64)
    ctx.check(ctx.lib.gatb_count_work(smp.handle, annos.handle, B, device._p(work)))
    segs, tested, n_entries, index_bytes = (int(x) for x in work)
    placed_per_sample = segs / float(B)
    mb = microbench(ctx.lib, local)
    hbm_peak, hbm_src = measured_peak()
    l2_bytes = 8.0 * pairs + 8.0 * segs + index_bytes
    hbm_bytes = index_bytes + 8.0 * segs + 4.0 * A * B
    ref_bytes = B * (8.0 * (A * placed_per_sample + wl["n_a_total"]) + 4.0 * A)
    sec = count_ms / 1000.0
    l2_peak = mb.get("l2_read_gbs")
    facts = ncu_facts() or {}
    roof = {"bound": "l2", "kernel": "count_kernel", "achieved": l2_bytes / sec / 1e9, "peak": l2_peak, "unit": "GB/s",
            "frac": (l2_bytes / sec / 1e9 / l2_peak) if l2_peak else None,
            "peak_source": "gatb_microbench: L2 read bandwidth measured in this run (48 MB buffer, 16-byte loads, all SMs)",
            "formula": "achieved = (8*pairs + 8*placed_segments + index_bytes) / kernel_ms; all per launch of `batch` samples",
            "kernel_ms": count_ms, "algorithmic_bytes_per_launch": l2_bytes,
            "work": {"batch": B, "placed_segments": segs, "overlapping_pairs": pairs, "entries_tested": tested,
                     "index_entries": n_entries, "index_bytes": index_bytes,
                     "pairs_per_segment": pairs / max(segs, 1), "entries_tested_per_segment": tested / max(segs, 1),
                     "tested_per_pair": tested / max(pairs, 1)},
            "hbm": {"achieved": hbm_bytes / sec / 1e9, "peak": hbm_peak, "frac": hbm_bytes / sec / 1e9 / hbm_peak,
                    "peak_source": hbm_src, "compulsory_bytes_per_launch": hbm_bytes},
            "traffic": (facts["dram_bytes_per_sample"] * B) if "dram_bytes_per_sample" in facts else None,
            "traffic_source": facts.get("capture"),
            "issue": None,
            "l1tex_data_pipe_pct_of_peak": facts.get("l1tex_throughput_pct"),     # (ncu capture: the unit that saturates)
            "reference_algorithm_equivalent": {"bytes_per_launch": ref_bytes, "GBps": ref_bytes / sec / 1e9,
                                               "x_hbm_peak": ref_bytes / sec / 1e9 / hbm_peak,
                                               "note": "SURVEY 8d: what the reference's per-cell two-pointer merge "
                                                       "streams; the index answers the same cells without it"},
            "kernel_share_of_step": prof["count"][0] / max(sum(v[0] for v in prof.values()), 1e-9),
            "other_kernels": {"place_kernel_ms": place_ms, "contig_merge_kernel_ms": merge_ms,
                              "place_algorithmic_GBps": 16.0 * segs / max(place_ms, 1e-9) / 1e6,
                              "placements_per_s": segs / max(place_ms, 1e-9) * 1e3}}
    if mb.get("issue_gwarp_inst_s") and facts.get("warp_instructions_per_launch") and \
            facts.get("samples_per_launch_in_capture") == B and facts.get("workload") == args.config:
        rate = facts["warp_instructions_per_launch"] / sec / 1e9
        roof["issue"] = {"achieved_gwarp_inst_s": rate, "peak_gwarp_inst_s": mb["issue_gwarp_inst_s"],
                         "frac": rate / mb["issue_gwarp_inst_s"],
                         "nominal_gwarp_inst_s": (4.0 * mb.get("sms", 0) * sm_mhz / 1e3) if sm_mhz else None,
                         "frac_of_nominal": (rate / (4.0 * mb.get("sms", 0) * sm_mhz / 1e3)) if (sm_mhz and mb.get("sms")) else None,
                         "warp_instructions_per_launch": facts["warp_instructions_per_launch"],
                         "source": facts.get("capture"),
                         "peak_source": "gatb_microbench: interleaved IADD3 / FFMA chains, 64 warps per SM, measured in this run "
                                        "(nominal 4 x %i SMs x clock)" % mb.get("sms", 0)}
    return roof, placed_per_sample


def stats_roofline(ctx, slab, S, A):
    """K5 (column statistics of the step's count matrix, resident in HBM) against the HBM roofline: the streaming
    passes of stats_stream.cu read the S x A uint32 matrix once each -- pass 1 plus one select pass per non-zero
    nibble of the largest count -- so achieved = passes * S * A * 4 bytes / kernel time (CUDA events around every
    launch, gatb_profile); peak = measured HBM copy bandwidth"""
    observed = slab[0].cpu().numpy().astype(np.float64)
    reps = 3
    ctx.column_stats(None, observed, device_ptr=slab.data_ptr(), n_samples=S, n_cols=A, is_float=False)     # warm-up
    ctx.profile(True)
    ctx.profile_read()
    for _ in range(reps):
        ctx.column_stats(None, observed, device_ptr=slab.data_ptr(), n_samples=S, n_cols=A, is_float=False)
    ms, launches = ctx.profile_read()["other"]
    ctx.profile(False)
    ms, launches = ms / reps, launches // reps
    passes = launches                               # (profiled scopes: pass 1 + one per select pass, each reads the matrix once)
    peak, src = measured_peak()
    gbs = passes * S * A * 4.0 / (ms / 1000.0) / 1e9
    return {"kernel": "stats_stream_kernel (K5 column statistics: TMA bulk copies into a shared-memory ring)",
            "bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak, "peak_source": src,
            "kernel_ms": ms, "passes_over_matrix": passes, "matrix_bytes": S * A * 4, "launches": launches,
            "formula": "achieved = passes * S * A * 4 / kernel_ms (the matrix of one step, %.0f MB, larger than L2)" % (S * A * 4 / 1e6)}


# --------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from gat_b200 import device

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries ONE JSON line: whatever libraries print there (NCCL's version banner, ...) is sent to
    # stderr by pointing file descriptor 1 at it; the JSON line goes to the saved descriptor at the end
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group(backend="cpu:gloo,cuda:nccl")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)

    wl = build_workload(args)
    pr, A, C, S = wl["problem"], wl["A"], wl["C"], args.samples_per_step
    cid = device.COUNTER_ID[args.counter]
    is_density = cid == device.DENSITY
    odt = torch.float64 if is_density else torch.int32

    ctx = device.Context(local)
    # a dedicated (non-default) stream: kernels, NCCL and the timing events all live on it; the legacy
    # default stream would add implicit synchronisation with every other stream
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    ctx.set_batch_size(args.batch)
    annos = device.Annotations(ctx, None, key_ws_nseg=wl["nseg"], csr=(A, C) + wl["anno_csr"])
    smp = device.Sampler(ctx, pr.unit_contig, C, pr.has_isochores, None, None, csr=(wl["seg_csr"], wl["ws_csr"]))
    # two output slabs, used alternately: for N > 1 the all-gather of step i (NCCL, asynchronous, its own stream)
    # overlaps the placement and counting of step i + 1, which write the other slab
    nbuf = 2 if (world > 1 or args.e2e_device_path) else 1
    peer = world > 1 and args.gather != "nccl" and not is_density
    if world > 1 and not peer:
        args.gather = "nccl"
    pending = [None] * nbuf
    if peer:
        # the gathered matrix of a step lives in memory every rank can write: each rank's counting kernels store
        # their rows into all of them (two matrices, used alternately like the NCCL slabs)
        from gat_b200 import parallel
        try:
            peers = [parallel.PeerMatrix(ctx, 1, world * S, A) for _ in range(nbuf)]
        except parallel.PeerUnavailable as e:      # (raised on every rank alike): the collective route instead
            sys.stderr.write("bench: %s -- falling back to --gather nccl\n" % e)
            peer, args.gather = False, "nccl"
    if peer:
        ctx.set_route_mode(args.gather == "peer-kernel")
        gathers = [pm.tensor[0] for pm in peers]
        outs = [g[rank * S:(rank + 1) * S] for g in gathers]
        routes = [[dict(base=pm.pointer(r), row_stride=A, row0=rank * S, col_begin=0, col_end=A) for r in range(world)]
                  for pm in peers]
    else:
        outs = [torch.zeros((S, A), dtype=odt, device=dev) for _ in range(nbuf)]
        gathers = [torch.empty((world * S, A), dtype=odt, device=dev) for _ in range(nbuf)] if world > 1 else None

    def run_into(t, begin, n):
        if is_density:
            return smp.run(annos, [args.counter], SEED, 0, begin, n, out_counts_ptr=None, out_density_ptr=t.data_ptr())
        return smp.run(annos, [args.counter], SEED, 0, begin, n, out_counts_ptr=t.data_ptr())

    def step_begin(i, r=None):
        return (i * world + (rank if r is None else r)) * S      # global sample indices of a rank's shard

    def step(i):
        b = i % nbuf
        if peer:                                   # the exchange is the kernels' epilogue: nothing to launch after them
            ctx.set_output_routes(routes[b])
            return run_into(outs[b], step_begin(i), S)
        if pending[b] is not None:                 # the slab's previous all-gather must have read it
            pending[b].wait()
            pending[b] = None
        info = run_into(outs[b], step_begin(i), S)
        if world > 1:
            pending[b] = dist.all_gather_into_tensor(gathers[b], outs[b], async_op=True)
        return info

    def drain():                                   # every all-gather in flight joins the launching stream
        for b in range(nbuf):
            if pending[b] is not None:
                pending[b].wait()
                pending[b] = None

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            box = [None] * world
            dist.all_gather_object(box, rank)      # (gloo: a barrier that launches nothing on the GPUs)
        torch.cuda.synchronize(dev)

    for i in range(args.warmup):
        info = step(i)
    drain()

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
        time.sleep(0.2)
    barrier()
    launches0 = ctx.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin = clocks.mark()
    e0.record(stream)
    for i in range(args.steps):
        info = step(args.warmup + i)
    drain()                                        # the last all-gathers are inside the timed region
    e1.record(stream)
    barrier()
    t_end = clocks.mark()
    ms = e0.elapsed_time(e1)
    launches = ctx.launch_count - launches0
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64)            # (host tensor: reduced over gloo)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    clock_info = clocks.stop(t_begin, t_end) if rank == 0 else None
    value = world * S * args.steps / (ms / 1000.0)
    last = args.warmup + args.steps - 1
    if args.dump_outputs:                          # (before the checks and profiled steps below reuse the slabs)
        if rank == 0:
            matrix = gathers[last % nbuf] if world > 1 else outs[last % nbuf]
            index = np.concatenate([step_begin(last, r) + np.arange(S) for r in range(world)])
            dump_outputs(args.dump_outputs, matrix, index)
        barrier()

    # ---- checks, outside the timed region: the slab of the last timed step against the CPU oracle, and (N > 1)
    # the gathered matrix of that step against a single-rank recomputation of every rank's global indices
    parity_check = gather_check = None
    if not args.no_checks:
        if rank == 0:
            from oracle import oracle as O
            slab = outs[last % nbuf]
            bad = []
            for row in (0, S - 1):
                exp = O.compute_sample_philox(pr.unit_contig, pr.unit_segments, pr.unit_workspace, wl["lists"],
                                              wl["nseg"], [args.counter], seed=SEED, track=0,
                                              sample=step_begin(last) + row, has_isochores=pr.has_isochores)[0]
                got = slab[row].cpu().numpy().astype(np.float64)
                if not np.array_equal(got, exp):
                    bad.append(row)
            parity_check = "ok" if not bad else "MISMATCH in rows %s" % bad
        if world > 1:
            if rank == 0:
                g = gathers[last % nbuf]
                tmp = torch.zeros((S, A), dtype=odt, device=dev)
                bad = []
                ctx.set_output_routes([])
                for r in range(world):
                    run_into(tmp, step_begin(last, r), S)
                    torch.cuda.synchronize(dev)
                    if not torch.equal(tmp, g[r * S:(r + 1) * S]):
                        bad.append(r)
                del tmp
                gather_check = "ok" if not bad else "MISMATCH for ranks %s" % bad
            barrier()

    # ---- per-kernel times (CUDA events around each launch, same stream), for the roofline
    ctx.profile(True)
    nprof = max(1, min(args.steps, 2))
    for i in range(nprof):
        step(last + 1 + i)
    drain()
    prof = ctx.profile_read()
    ctx.profile(False)
    ctx.set_output_routes([])
    roofline, placed_per_sample = (None, float(info[0]) / S)
    if rank == 0:
        roofline, placed_per_sample = roofline_of(args, wl, ctx, smp, annos, prof, local,
                                                  sm_mhz=(clock_info or {}).get("sm_mhz"))
        if odt == torch.int32 and not args.no_checks:
            try:
                roofline["statistics_kernel"] = stats_roofline(ctx, outs[last % nbuf], S, A)
            except Exception as exc:               # (reported, never fatal for the headline)
                roofline["statistics_kernel"] = {"error": str(exc)}
    barrier()

    # ---- e2e: host buffers in, host count matrix out, through the C ABI, every step
    e2e = None
    if not args.no_e2e:
        def pinned(x):       # pinned copies of the CSR buffers (viewed signed: torch lacks some unsigned ops)
            signed = {np.dtype(np.uint64): np.int64, np.dtype(np.uint32): np.int32}[x.dtype]
            return torch.from_numpy(np.ascontiguousarray(x).view(signed)).pin_memory()

        pin = [pinned(x) for x in wl["anno_csr"] + wl["seg_csr"] + wl["ws_csr"]]
        unsign = {torch.int64: np.uint64, torch.int32: np.uint32}
        pa = tuple(t.numpy().view(unsign[t.dtype]) for t in pin[0:3])
        ps = tuple(t.numpy().view(unsign[t.dtype]) for t in pin[3:6])
        pw = tuple(t.numpy().view(unsign[t.dtype]) for t in pin[6:9])
        h2d = sum(t.numel() * t.element_size() for t in pin)
        host_outs = [torch.empty((S, A), dtype=odt).pin_memory() for _ in range(nbuf)]
        host_out = host_outs[0]
        host_np = host_out.numpy()
        side = torch.cuda.Stream(device=dev)
        copied = [None] * nbuf
        ids = device.counter_ids([args.counter])
        info_np = np.zeros(3, dtype=np.uint64)

        def e2e_upload():
            # gatb_annotations_create_async returns once the copies from the pinned host arrays and the index
            # build are queued on the context's upload / build streams
            return device.Annotations(ctx, None, key_ws_nseg=wl["nseg"], csr=(A, C) + pa, lazy=True)

        def e2e_steps(first, n):
            # Double-buffered: EVERY step uploads its own copy of all inputs and reads its count matrix back to
            # the host, but the annotation upload + index build of step i+1 are queued before gatb_run of step
            # i, so they overlap its placement and counting kernels (copy engine + build stream next to the
            # compute stream); gatb_run(i) only waits for ITS set before launching the count.  The first
            # step's upload is not hidden behind anything and is inside the timed region like the others.
            tm = collections.Counter()
            clock = [time.perf_counter()]

            def lap(name):                          # host-side phase times of the loop (GATB_BENCH_TRACE=1: on stderr)
                now = time.perf_counter()
                tm[name] += now - clock[0]
                clock[0] = now

            nxt = e2e_upload()
            lap("upload")
            for j in range(n):
                # (the sampler first: its small uploads and read-backs must not queue behind the next step's 159 MB of
                # annotation arrays on the copy engine)
                s2 = device.Sampler(ctx, pr.unit_contig, C, pr.has_isochores, None, None, csr=(ps, pw))
                lap("sampler")
                a2, nxt = nxt, (e2e_upload() if j + 1 < n else None)
                lap("upload")
                begin = step_begin(first + j)
                if world == 1 and not args.e2e_device_path:
                    # host in, host out: gatb_run copies every batch's counts to the pinned host matrix while
                    # the next batch is being placed and counted
                    ctx.check(ctx.lib.gatb_run(s2.handle, a2.handle, 1, device._p(ids), SEED, 0, begin, S,
                                               None if is_density else device._p(host_np.view(np.uint32)),
                                               device._p(host_np) if is_density else None, 0, device._p(info_np)))
                elif peer:
                    # N > 1, peer exchange: one gatb_run delivers every batch's rows to the pinned host matrix AND, through
                    # the output routes, to every rank's device matrix (copy engines, behind the next batch's kernels)
                    b = j % nbuf
                    ctx.set_output_routes(routes[b])
                    ctx.check(ctx.lib.gatb_run(s2.handle, a2.handle, 1, device._p(ids), SEED, 0, begin, S,
                                               device._p(host_outs[b].numpy().view(np.uint32)), None, 0, device._p(info_np)))
                    lap("run")
                    barrier()               # every rank's rows have arrived in every matrix
                    lap("exchange")
                else:
                    # N > 1, NCCL: counts stay on the device for the all-gather; every rank then reads ITS rows of the
                    # gathered matrix back to the host -- on a side stream, while the next step already runs
                    # (two device matrices and two pinned host matrices, used alternately)
                    b = j % nbuf
                    if copied[b] is not None:
                        copied[b].synchronize()     # the copy that last read this matrix / wrote this host buffer
                    lap("wait copy")
                    ctx.check(ctx.lib.gatb_run(s2.handle, a2.handle, 1, device._p(ids), SEED, 0, begin, S,
                                               None if is_density else outs[b].data_ptr(),
                                               outs[b].data_ptr() if is_density else None, 1, device._p(info_np)))
                    lap("run")
                    if world > 1:
                        dist.all_gather_into_tensor(gathers[b], outs[b])
                    lap("exchange")
                    side.wait_stream(torch.cuda.current_stream(dev))
                    with torch.cuda.stream(side):
                        src = gathers[b][rank * S:(rank + 1) * S] if world > 1 else outs[b]
                        # (batch-sized pieces: one 393 MB copy would hold the device-to-host engine for 8 ms, and
                        # the next step's small read-backs -- unit descriptors, validation words -- queue behind it)
                        for k in range(0, S, args.batch):
                            host_outs[b][k:k + args.batch].copy_(src[k:k + args.batch], non_blocking=True)
                        copied[b] = torch.cuda.Event()
                        copied[b].record(side)
                lap("run" if world == 1 else "read-back queue")
                s2.close()
                a2.close()
                lap("close")
            for ev in copied:
                if ev is not None:
                    ev.synchronize()
            lap("wait copy")
            if os.environ.get("GATB_BENCH_TRACE") and rank == 0:
                sys.stderr.write("e2e host phases over %i steps (ms per step): %s\n"
                                 % (n, ", ".join("%s %.2f" % (k, 1e3 * v / n) for k, v in tm.items())))
            return int(host_np.reshape(-1)[:1].view(np.uint8)[0])

        if world == 1 and not args.e2e_device_path:
            ctx.set_stream(None)                    # host in / host out: the context's own stream
        # (step indices continue after the device-resident steps: global sample indices stay far below 2^32)
        e2e_first = last + 8
        e2e_steps(e2e_first, 2)                     # warm-up (allocator pools, pinned paths)
        barrier()
        t0 = time.perf_counter()
        e2e_steps(e2e_first + 2, args.steps)
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        e2e = {"value": world * S * args.steps / dt, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(S * A * (8 if is_density else 4)),
               "what": "per step of %i samples per GPU: gatb_sampler_create + gatb_annotations_create_async (every input "
                       "from pinned host memory, on every rank) + gatb_run%s + the step's count matrix read back to "
                       "pinned host memory; double-buffered: the upload + index build of step i+1 overlap the "
                       "kernels of step i" % (S, (" (host output AND output routes into every rank's peer matrix) + barrier" if peer else
                                                  " + NCCL all-gather of the slab + side-stream read-back") if world > 1 else
                                              " (host output: the copy of batch i overlaps batch i+1)")}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import ref_bench
        if ref_bench.available():
            rate, cores, sample = reference_rate(args, wl)
            cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample}
        else:
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": "oracle/_ref not built"}

    if rank == 0:
        line = {"metric": args.metric, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64" if is_density else "u32",
                "data": "synthetic", "config": config_of(args, wl, world), "clocks": clock_info,
                "e2e": e2e, "gpu_launches": int(launches), "parity_check": parity_check,
                "gather_check": gather_check, "roofline": roofline, "cpu_baseline": cpu,
                "placed_segments_per_sample": placed_per_sample,
                "segment_placements_per_s": value * placed_per_sample}
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    ctx.set_output_routes([])
    smp.close()
    annos.close()
    if world > 1:
        barrier()
        if peer:
            del gathers, outs
            for pm in peers:
                pm.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    if parity_check not in (None, "ok") or gather_check not in (None, "ok"):
        sys.exit(3)


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
