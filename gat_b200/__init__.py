"""gat_b200 -- B200-native simulation engine of the Genomic Association Tester.

Drop-in for the `gat.run()` / gat-run.py path of AndreasHeger/gat (gat/__init__.py:855-1088): same
arguments, same result objects, same output table.  The per-sample work of the reference
(UnconditionalSampler.sample -> computeSample, gat/__init__.py:494-591, 704-778) is replaced by batched
CUDA kernels reached through the C ABI in include/gat_b200.h.  One process per GPU; with
torch.distributed initialised the samples are sharded by rank and the count matrix is all-gathered
(gat_b200/parallel.py).
"""
import collections
import os
import re
import sys
import time

import numpy as np

from . import device
from . import engine as Engine
from . import matrixfree
from . import stats as Stats
from .engine import (IntervalCollection, IntervalDictionary, SamplerAnnotator, SamplerSegments, SamplerShift, UnconditionalWorkspace,
                     AnnotatorResult, AnnotatorResultExtended, getContext, seed)
from .segmentlist import SegmentList

__version__ = "0.1.0"


class TrackProblem(object):
    """one segment track flattened for the GPU: placement units in the reference's iteration order and
    the contig-level annotations/workspace they are counted against."""

    def __init__(self, segs, workspace):
        # units = keys of the track in iteration order, skipping empty ones (gat/__init__.py:531-538)
        self.unit_keys = []
        self.contigs = []
        contig_index = {}
        self.unit_contig = []
        self.has_isochores = False
        for key in list(segs.keys()):
            if workspace[key].isEmpty or segs[key].isEmpty:
                continue
            contig, split = Engine.splitKey(key)
            self.has_isochores = self.has_isochores or split
            if contig not in contig_index:
                contig_index[contig] = len(self.contigs)
                self.contigs.append(contig)
            self.unit_keys.append(key)
            self.unit_contig.append(contig_index[contig])
        self.unit_segments = [segs[k].asarray() for k in self.unit_keys]
        self.unit_workspace = [workspace[k].asarray() for k in self.unit_keys]


def buildContigAnnotations(annotations, workspace, contigs):
    """contig-level annotations and workspace as UnconditionalSampler.sample builds them
    (gat/__init__.py:716-721): clone + fromIsochores; lists[a][c] and len(contig_workspace[c])"""
    contig_annotations = annotations.clone()
    contig_annotations.fromIsochores()
    contig_workspace = workspace.clone()
    contig_workspace.fromIsochores()
    atracks = list(annotations.tracks)
    lists = [[contig_annotations[a][c].asarray() for c in contigs] for a in atracks]
    nseg = [len(contig_workspace[c]) for c in contigs]
    return atracks, lists, nseg


def trackSampler(segs, annotations, workspace, sampler, annos_cache=None):
    """the GPU objects that sample one track: -> (smp, annos), device.Sampler and device.Annotations, or
    (None, None) for a track without any unit (every sample counts zero)"""
    ctx = getContext()
    problem = TrackProblem(segs, workspace)
    if not problem.unit_keys:
        return None, None
    try:
        smp = device.Sampler(ctx, problem.unit_contig, len(problem.contigs), problem.has_isochores,
                             problem.unit_segments, problem.unit_workspace,
                             bucket_size=sampler.bucket_size, nbuckets=sampler.nbuckets)
    except device._lib.GatB200Error as e:
        if e.code == device._lib.ERR_TOO_LARGE:
            raise ValueError(str(e))
        raise
    if getattr(sampler, "kind", "annotator") == "shift":
        smp.set_shift(sampler.radius, sampler.extension)
    elif getattr(sampler, "kind", "annotator") != "annotator":
        try:
            smp.set_kind(sampler.kind)
        except device._lib.GatB200Error as e:
            raise AssertionError(str(e))       # the reference's counters assert on unnormalized samples
    # (the sampler first: its small uploads must not queue behind the annotation arrays on the copy
    # engine; the annotations then upload and build while the placement kernel runs)
    key = tuple(problem.contigs)
    if annos_cache is not None and key in annos_cache:
        annos = annos_cache[key]
    elif not problem.has_isochores:
        # no isochores: fromIsochores changes nothing, the contig-level annotations are the loaded ones
        annos, _ = Engine.deviceAnnotations(annotations, problem.contigs, [len(workspace[c]) for c in problem.contigs],
                                            annos_cache, lazy=True)
    elif getattr(annotations, "onDevice", False):
        # isochores, lists on the GPU: clone + fromIsochores there (gat/__init__.py:716-721), index built in place
        contig_annotations = annotations.clone()
        contig_annotations.fromIsochores()
        contig_workspace = workspace.clone()
        contig_workspace.fromIsochores()
        annos, _ = Engine.deviceAnnotations(contig_annotations, problem.contigs,
                                            [len(contig_workspace[c]) for c in problem.contigs], annos_cache)
        contig_annotations._drop_device()
    else:
        _, lists, nseg = buildContigAnnotations(annotations, workspace, problem.contigs)
        annos = device.Annotations(ctx, lists, key_ws_nseg=nseg, lazy=True)
        if annos_cache is not None:
            annos_cache[key] = annos
    return smp, annos


RunPlan = collections.namedtuple("RunPlan", "exchange transport matrix_free rows columns")

# one track's samples after the exchange: per counter the plane this rank holds (Engine.SampleMatrix; float64 for
# density) or the finished statistics (matrix-free), and whether the statistics of its columns must be gathered
TrackSamples = collections.namedtuple("TrackSamples", "atracks planes gather")

# the inputs of one run(): observed[counter_id] = {track: {annotation: count}}
# (shard: None, or the (begin, end) sample range of a shard job)
_Job = collections.namedtuple("_Job", "segments annotations workspace sampler counters observed reference num_samples "
                                      "pseudo_count samples_pattern annos_cache shard")

_STATS = ("expected", "stddev", "lower95", "upper95", "fold", "pvalue")


def run(segments, annotations, workspace, sampler, counters, workspace_generator, **kwargs):
    """run an enrichment analysis (signature and kwargs of gat.run, gat/__init__.py:855-907).

    kwargs: num_samples (10000), pseudo_count (1.0), reference, output_counts_pattern,
    output_samples_pattern, outfiles, cache / sample_files / num_threads (accepted, unused: the
    reference's sample cache is dead code and its multiprocessing is replaced by the GPU);
    exchange ("auto" | "allgather" | "columns"), transport ("peer" | "nccl"): how a multi-GPU run combines its slabs;
    keep_samples (None | True | False): False computes the statistics without the sample matrix
    (gat_b200/matrixfree.py), so that the number of samples is not bounded by GPU memory -- the results are the
    same, but their samples cannot be asked for; None (default) does so only when the matrices would not fit in
    the free GPU memory and no counts table is written.
    """
    return _onRunStream(_run, segments, annotations, workspace, sampler, counters, workspace_generator, **kwargs)


def runShard(segments, annotations, workspace, sampler, counters, workspace_generator, sample_range, filename, **kwargs):
    """one shard of a run: the global samples [begin, end) = sample_range of run(..., num_samples=...) with the same
    arguments (kwargs of run()), written to `filename` as the exact integer state of every (track, counter) instead of
    statistics (gat_b200/shards.py).  Shards of the same inputs and seed whose ranges tile [0, num_samples) merge, in
    any order, into run()'s results bit for bit (mergeShards).  The run must be seeded (engine.seed): each shard
    would otherwise draw a seed of its own.  On several ranks each rank samples its part of the range and rank 0
    writes the file.  Returns None."""
    _onRunStream(_run, segments, annotations, workspace, sampler, counters, workspace_generator,
                 shard=(tuple(sample_range), filename), **kwargs)


def _onRunStream(fn, *args, **kwargs):
    import torch
    # ONE CUDA stream for the whole run: the library's kernels, torch's tensor operations and the NCCL
    # collectives are all ordered on it (the library's own stream is non-blocking: it would not even wait for
    # torch's default stream)
    ctx = getContext()
    dev = torch.device("cuda", ctx.device)
    stream = torch.cuda.Stream(device=dev)
    stream.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(stream):
        try:
            return fn(*args, **kwargs)
        finally:
            torch.cuda.synchronize(dev)
            ctx.set_stream(None)


def _planRun(num_samples, n_tracks, n_annotations, counter_names, counts_table, keep_samples, exchange, transport,
             rank, world, free_bytes, sample_range=None, seeded=True):
    """how run() computes, from sizes alone (no I/O, no collective, no device query) -> RunPlan; every refusal of
    a bad argument is made here, alike on every rank and before the run's first collective.

    exchange: how the per-rank slabs [S/G][A] become statistics (SURVEY 8e / 8f2).  "allgather": every rank holds
      the S x A matrix.  "columns": rank g holds all S samples of ITS A/G columns and only the <= 6 x A result doubles
      are gathered, 1/G of the traffic and memory.  "auto": columns once the gathered matrices would exceed 1 GiB per
      rank, unless a counts table (every column on rank 0) is wanted.
    transport: "peer" -- the counting kernels store every finished row straight into the destination ranks' matrices
      (CUDA IPC, output routes of the C ABI), no collective follows; integer counters only.  "nccl" -- one NCCL
      collective per counter plane after the kernels.
    matrix_free: stream the samples through column accumulators instead of keeping the S x A matrices; exchange and
      transport do not apply then.  free_bytes (keep_samples=None only) differs between GPUs: run() makes them agree.
    rows, columns: [begin, end) of this rank's global sample indices and of the annotation columns it holds.
    sample_range: (begin, end) of a shard job (runShard): its rows are this rank's part of the range, always counted
      by the matrix-free accumulators; seeded: a seed was set before the run (a shard must not draw its own)."""
    from . import parallel
    if sample_range is not None:
        return _planShard(num_samples, n_annotations, counter_names, counts_table, keep_samples, rank, world,
                          sample_range, seeded)
    if exchange not in ("auto", "allgather", "columns"):
        raise ValueError("exchange must be auto, allgather or columns")
    if exchange == "auto":
        big = 4 * num_samples * n_annotations * len(counter_names) >= (1 << 30)
        exchange = "columns" if (world > 1 and big and not counts_table) else "allgather"
    if world == 1:
        exchange = "allgather"
    if exchange == "columns" and counts_table:
        raise ValueError("output_counts_pattern needs every column on rank 0: use exchange='allgather'")
    columns = _columnRange(exchange, n_annotations, rank, world)
    density = "nucleotide-density" in counter_names
    matrix_bytes = 4 * len(counter_names) * num_samples * (columns[1] - columns[0]) * n_tracks
    matrix_free = matrixfree.use_matrix_free(keep_samples, counts_table, density, matrix_bytes, free_bytes)
    if transport not in ("peer", "nccl"):
        raise ValueError("transport must be peer or nccl")
    if world == 1 or density:
        transport = "nccl"              # (one rank: nothing to exchange; the float64 density plane is not routed)
    return RunPlan(exchange, transport, matrix_free, parallel.shard_range(num_samples, rank, world), columns)


def _planShard(num_samples, n_annotations, counter_names, counts_table, keep_samples, rank, world, sample_range,
               seeded):
    from . import parallel
    begin, end = (int(x) for x in sample_range)
    if counts_table:
        raise ValueError("a shard job writes no counts table: output_counts_pattern needs every sample in one run")
    if keep_samples:
        raise ValueError("a shard job keeps no samples: keep_samples=True is refused")
    if not 0 <= begin < end <= num_samples < (1 << 32):
        raise ValueError("sample_range (%i, %i) must satisfy 0 <= begin < end <= num_samples (%i) < 2^32"
                         % (begin, end, num_samples))
    if "nucleotide-density" in counter_names:
        raise NotImplementedError("nucleotide-density has no shard mode (float64 samples have no exact split)")
    if not seeded:
        raise ValueError("a shard job needs a seeded run (engine.seed, --random-seed): every shard must place the "
                         "same samples")
    b, e = parallel.shard_range(end - begin, rank, world)
    return RunPlan("allgather", "nccl", True, (begin + b, begin + e), (0, n_annotations))


def _columnRange(exchange, n_annotations, rank, world):
    from . import parallel
    return parallel.column_range(n_annotations, rank, world) if exchange == "columns" else (0, n_annotations)


def _run(segments, annotations, workspace, sampler, counters, workspace_generator, shard=None, **kwargs):
    """run() -> results; runShard() (shard = (sample_range, filename)) -> None, the shard file written"""
    from . import parallel
    import torch
    num_samples = kwargs.get("num_samples", 10000)
    output_counts_pattern = kwargs.get("output_counts_pattern", None)
    keep_samples = kwargs.get("keep_samples", None)
    if not getattr(sampler, "accelerated", False):
        raise NotImplementedError("sampler %s is not accelerated by gat_b200 (only SamplerAnnotator is)"
                                  % type(sampler).__name__)
    if getattr(workspace_generator, "is_conditional", False):
        raise NotImplementedError("conditional workspaces are not accelerated by gat_b200")

    ctx = getContext()
    rank, world = parallel.rank_world()
    parallel.join_warm_up()
    seconds, last = ({} if os.environ.get("GATB_TIMING") else None), [time.perf_counter()]

    def mark(name):                     # GATB_TIMING=1: seconds per phase, each summed over the tracks
        if seconds is not None:
            torch.cuda.synchronize(ctx.device)
            now = time.perf_counter()
            seconds[name] = seconds.get(name, 0.0) + now - last[0]
            last[0] = now

    # observed counts (gat/__init__.py:932-940)
    annos_cache = {}      # key tuple -> device.Annotations: one upload + index build per key set for the whole run
    observed = [Engine.computeCounts(counter=c, aggregator=sum, segments=segments, annotations=annotations,
                                     workspace=workspace, workspace_generator=workspace_generator,
                                     annos_cache=annos_cache) for c in counters]
    mark("observed")
    job = _Job(segments, annotations, workspace, sampler, counters, observed, kwargs.get("reference", None),
               num_samples, kwargs.get("pseudo_count", 1.0), kwargs.get("output_samples_pattern", None), annos_cache,
               None if shard is None else shard[0])

    free_bytes = torch.cuda.mem_get_info(ctx.device)[0] if keep_samples is None else 0
    n_annotations = len(list(annotations.tracks))
    plan = _planRun(num_samples, len(segments.tracks), n_annotations, [c.name for c in counters],
                    bool(output_counts_pattern), keep_samples,
                    kwargs.get("exchange", os.environ.get("GATB_EXCHANGE", "auto")),
                    kwargs.get("transport", os.environ.get("GATB_TRANSPORT", "peer")), rank, world, free_bytes,
                    sample_range=job.shard, seeded=Engine._rng_state["seed"] is not None)
    # every rank must place with the SAME seed (the matrix is keyed by seed and global sample index): an
    # unseeded run draws its seed on rank 0 and broadcasts it
    parallel.share_seed()
    if keep_samples is None and world > 1 and shard is None:
        plan = plan._replace(matrix_free=any(matrixfree.allgather(plan.matrix_free, world)))

    # (torch's legacy default stream has handle 0 = "the library's own stream" at the C ABI: pass cudaStreamLegacy)
    ctx.set_stream(torch.cuda.current_stream(ctx.device).cuda_stream or 1)
    slab = _matrixFreeSlab(len(counters), n_annotations, plan) if plan.matrix_free else None
    sampled = {}
    for ntrack, track in enumerate(segments.tracks if workspace.sum() > 0 else ()):
        peer, plan = _peerMatrix(plan, len(counters), num_samples)
        sampled[track] = _sampleTrack(ntrack, track, job, plan, peer, slab, mark)

    sizes = _sizes(job, sampled)
    for a in annos_cache.values():
        a.close()
    mark("overlap columns")
    if shard is not None:
        if rank == 0:
            from . import shards
            shards.writeShard(shard[1], job, sampled, sizes)
        mark("shard file")
        if seconds is not None and rank == 0:
            sys.stderr.write("# gat_b200.runShard phases: " + ", ".join("%s %.3fs" % p for p in seconds.items()) + "\n")
        return None

    # statistics per (counter, track): one batched column-stats call over all annotations
    results = []
    for counter_id, counter in enumerate(counters):
        for track, r in job.observed[counter_id].items():
            if track in sampled:
                st, matrix = _statistics(job, sampled[track], counter_id, track)
                results.extend(_results(job, track, counter.name, r, sampled[track].atracks, st, matrix, sizes))
    if output_counts_pattern and rank == 0:
        _writeCounts(output_counts_pattern, counters, results)
    torch.cuda.synchronize(ctx.device)
    mark("statistics+results")
    if seconds is not None and rank == 0:
        sys.stderr.write("# gat_b200.run phases: " + ", ".join("%s %.3fs" % p for p in seconds.items()) + "\n")
    return results


def _peerMatrix(plan, n_counters, num_samples):
    """-> (PeerMatrix or None, plan): every rank's destination matrix of the peer transport, writable by all:
    [counter][S][all columns | its own columns].  When the GPUs cannot map each other's memory (every rank alike),
    the rest of the run takes the NCCL transport."""
    from . import parallel
    if plan.transport != "peer" or plan.matrix_free:
        return None, plan
    try:
        return parallel.PeerMatrix(getContext(), n_counters, num_samples, max(plan.columns[1] - plan.columns[0], 1)), plan
    except parallel.PeerUnavailable as e:
        if parallel.rank_world()[0] == 0:
            sys.stderr.write("# gat_b200.run: %s -- using the NCCL transport\n" % e)
        return None, plan._replace(transport="nccl")


def _matrixFreeSlab(n_counters, n_annotations, plan):
    """the one device buffer every slab of the matrix-free mode is counted into -> (int32 tensor, rows per slab)"""
    import torch
    matrixfree.info.update(reruns=0, arena_bytes=0, chunk_rows=0, pass2_seconds=0.0)
    n_local = plan.rows[1] - plan.rows[0]
    chunk = max(1, min(max(n_local, 1), matrixfree.SLAB_BYTES // (4 * n_counters * max(n_annotations, 1))))
    return torch.zeros(n_counters * chunk * max(n_annotations, 1), dtype=torch.int32, device=getContext().device), chunk


def _sampleTrack(ntrack, track, job, plan, peer, slab, mark):
    """all samples of one track (replaces UnconditionalSampler.sample, gat/__init__.py:704-778), exchanged between
    the ranks -> TrackSamples.  A track without any unit counts zero in every sample: a zero plane of all columns on
    every rank, or zero slabs in the matrix-free mode."""
    import torch
    from . import parallel
    atracks = list(job.annotations.tracks)
    names = [c.name for c in job.counters]
    smp, annos = trackSampler(job.segments[track], job.annotations, job.workspace, job.sampler, job.annos_cache)
    try:
        if plan.matrix_free:
            stats = _streamTrack(ntrack, track, smp, annos, names, atracks, job, plan, slab)
        elif smp is not None:
            out_u, out_f = _sampleRows(ntrack, smp, annos, names, len(atracks), plan, peer)
        if smp is not None and job.samples_pattern and parallel.rank_world()[0] == 0:
            _dumpSamples(smp, track, ntrack, job.segments[track], job.workspace, job.num_samples, job.samples_pattern)
    finally:
        if smp is not None:
            smp.close()
    mark("sampling")
    if plan.matrix_free:
        return TrackSamples(atracks, stats, False)
    if smp is None:
        if peer is not None:
            parallel.barrier()
            peer.close()
        zeros = torch.zeros((job.num_samples, len(atracks)), dtype=torch.int32, device=getContext().device)
        return TrackSamples(atracks, [Engine.SampleMatrix(zeros, True) for _ in names], False)
    out_u, out_f = _exchange(out_u, out_f, peer, plan, job.num_samples)
    mark("exchange")
    planes = [Engine.SampleMatrix(out_f if name == "nucleotide-density" else out_u[i], name != "nucleotide-density",
                                  first_column=plan.columns[0]) for i, name in enumerate(names)]
    return TrackSamples(atracks, planes, plan.exchange == "columns")


def _sampleRows(ntrack, smp, annos, names, n_annotations, plan, peer):
    """this rank's rows of the track -> (int32 [counters][rows][A], float64 [rows][A] of the density counter or None).
    With a PeerMatrix the counting kernels deliver the rows straight to every rank's matrix (output routes,
    device.Context.set_output_routes) instead: -> (None, None)"""
    import torch
    ctx = getContext()
    begin, end = plan.rows
    if peer is not None:
        routes = []
        for r in range(peer.world):
            cb, ce = _columnRange(plan.exchange, n_annotations, r, peer.world)
            _, rows_r, cols_r = peer.shape_of(r)
            if ce > cb:
                routes.append(dict(base=peer.pointer(r), plane_stride=rows_r * cols_r, row_stride=cols_r, row0=begin,
                                   col_begin=cb, col_end=ce))
        if end > begin:
            ctx.set_output_routes(routes)
            try:
                smp.run(annos, names, Engine.getSeed(), ntrack, begin, end - begin, out_counts_ptr=routes[0]["base"])
            finally:
                ctx.set_output_routes([])
        return None, None
    out_u = torch.zeros((len(names), max(end - begin, 1), n_annotations), dtype=torch.int32, device=ctx.device)
    out_f = torch.zeros((max(end - begin, 1), n_annotations), dtype=torch.float64, device=ctx.device) \
        if "nucleotide-density" in names else None
    smp.run(annos, names, Engine.getSeed(), ntrack, begin, end - begin,
            out_counts_ptr=out_u.data_ptr(), out_density_ptr=out_f.data_ptr() if out_f is not None else None)
    return out_u, out_f


def _exchange(out_u, out_f, peer, plan, num_samples):
    """every rank's slabs -> (out_u, out_f) of all S samples of this rank's columns"""
    import torch
    from . import parallel
    begin, end = plan.rows
    if peer is not None:
        parallel.barrier()              # every rank's kernels have delivered their rows
        out_u = peer.tensor[:, :, :plan.columns[1] - plan.columns[0]].clone()
        parallel.barrier()              # (nobody frees memory a peer still has mapped for writing)
        peer.close()
    elif plan.exchange == "columns":
        # one collective per counter plane: all-to-all by column
        planes = [parallel.exchange_columns(out_u[i][:end - begin], num_samples) for i in range(out_u.shape[0])]
        out_u = torch.stack(planes) if planes else out_u
        if out_f is not None:
            out_f = parallel.exchange_columns(out_f[:end - begin], num_samples)
    else:
        # one collective: all-gather the S/G x A slabs of every counter (SURVEY 8e)
        out_u = parallel.allgather_samples(out_u, num_samples, dim=1)
        if out_f is not None:
            out_f = parallel.allgather_samples(out_f, num_samples, dim=0)
    return out_u, out_f


def _streamTrack(ntrack, track, smp, annos, names, atracks, job, plan, slab):
    """the matrix-free mode: this rank's samples in slabs of one reused device buffer, counted into column
    accumulators and overwritten -> [statistics dict per counter], complete (summed over the ranks); in a shard job
    [integer state per counter] of the shard's rows (matrixfree.shard_states)"""
    from . import parallel
    buf, chunk = slab
    begin, end = plan.rows

    def produce(r0, n):
        if smp is None:
            buf[:len(names) * n * len(atracks)].zero_()
        else:
            smp.run(annos, names, Engine.getSeed(), ntrack, begin + r0, n, out_counts_ptr=buf.data_ptr())
        return buf.data_ptr()

    rank, world = parallel.rank_world()
    planes = [_observed(job, counter_id, track, atracks) for counter_id in range(len(names))]
    if job.shard is not None:
        return matrixfree.shard_states(getContext(), produce, planes, job.num_samples, end - begin, len(atracks), chunk,
                                       rank=rank, world=world)
    return matrixfree.stream_statistics(getContext(), produce, planes, job.num_samples, end - begin, len(atracks), chunk,
                                        pseudo_count=job.pseudo_count, rank=rank, world=world)


def _observed(job, counter_id, track, atracks):
    """(observed values, reference folds or None) of one (counter, track), in the order of the annotation tracks"""
    r = job.observed[counter_id][track]
    ref = np.array([job.reference[track][a].fold for a in atracks], dtype=np.float64) if job.reference else None
    return np.array([r[a] for a in atracks], dtype=np.float64), ref


def _statistics(job, samples, counter_id, track):
    """-> (statistics dict of every annotation column, the samples the results hand out)"""
    import torch
    from . import parallel
    plane = samples.planes[counter_id]
    if isinstance(plane, dict):
        return plane, Engine.SamplesNotKept(job.num_samples, len(samples.atracks))
    # the plane stays on the GPU; column-sharded, it holds this rank's columns [first_column, first_column + ncolumns)
    obs, ref = _observed(job, counter_id, track, samples.atracks)
    lo, hi = plane.first_column, plane.first_column + plane.ncolumns
    if hi == lo:                        # more ranks than columns: nothing to do here
        st = dict((k, np.zeros(0)) for k in _STATS)
    else:
        st = getContext().column_stats(None, obs[lo:hi], pseudo_count=job.pseudo_count,
                                       ref_fold=None if ref is None else ref[lo:hi], device_ptr=plane._tensor.data_ptr(),
                                       n_samples=job.num_samples, n_cols=hi - lo, is_float=0 if plane._as_uint32 else 1)
    if samples.gather:
        # the result doubles of every rank's columns: one small all-gather
        # (host tensors: a few kB over the gloo side of the process group -- no NCCL set-up for this)
        full = parallel.allgather_columns(torch.from_numpy(np.stack([st[k] for k in _STATS])), len(obs)).numpy()
        st = dict((k, full[i]) for i, k in enumerate(_STATS))
    return st, plane


def _sizes(job, sampled):
    """size / overlap columns of AnnotatorResultExtended: once per track and per annotation, the overlap of a
    track with every annotation in one GPU call (gat/Engine.pyx:1911-1928 does one intersect per result)"""
    anno_sizes = job.annotations.trackSizes() if getattr(job.annotations, "onDevice", False) else \
        dict((a, (job.annotations[a].counts(), job.annotations[a].sum())) for a in job.annotations.tracks)
    track_sizes = {}
    for track in sampled:
        track_sizes[track] = (job.segments[track].counts(), job.segments[track].sum(),
                              Engine.overlapColumns(job.segments[track], job.annotations, job.annos_cache))
    return anno_sizes, track_sizes, job.workspace.sum()


def _results(job, track, counter, r, atracks, st, matrix, sizes):
    """the AnnotatorResultExtended of one (counter, track), in the order of the annotation tracks"""
    anno_sizes, track_sizes, workspace_size = sizes
    on_device = getattr(job.annotations, "onDevice", False)
    out = []
    for ai, annotation in enumerate(atracks):
        out.append(AnnotatorResultExtended(
            track=track, annotation=annotation, counter=counter, observed=r[annotation],
            samples=(matrix, ai), track_segments=job.segments[track],
            annotation_segments=None if on_device else job.annotations[annotation], workspace=job.workspace,
            reference=job.reference[track][annotation] if job.reference else None,
            pseudo_count=job.pseudo_count, stats=dict((k, float(v[ai])) for k, v in st.items()),
            sizes=dict(track_nsegments=track_sizes[track][0], track_size=track_sizes[track][1],
                       annotation_nsegments=anno_sizes[annotation][0], annotation_size=anno_sizes[annotation][1],
                       overlap_nsegments=track_sizes[track][2][annotation][0],
                       overlap_size=track_sizes[track][2][annotation][1], workspace_size=workspace_size)))
    return out


def _writeCounts(pattern, counters, results):
    """dump (large) table with counts (gat/__init__.py:1072-1086).  The reference formats every sample with "%i" in
    a Python loop; here the text of a whole S x A matrix comes from one GPU call (gatb_format_counts)"""
    for counter in counters:
        texts = {}                    # id(SampleMatrix) -> (text, column offsets)
        with _open(re.sub("%s", counter.name, pattern), "w") as outfile:
            outfile.write("track\tannotation\tobserved\tcounts\n")
            for o in results:
                if o.counter != counter.name:
                    continue
                matrix, ai = o._lazy
                if matrix._as_uint32:
                    if id(matrix) not in texts:
                        texts[id(matrix)] = matrix.text()
                    text, off = texts[id(matrix)]
                    column = text[int(off[ai]):int(off[ai + 1])].tobytes().decode("ascii")
                else:
                    column = ",".join(["%i" % x for x in o.samples])
                outfile.write("%s\t%s\t%i\t%s\n" % (o.track, o.annotation, o.observed, column))


def _open(filename, mode):
    import gzip
    if filename.endswith(".gz"):
        return gzip.open(filename, mode + "t")
    return open(filename, mode)


def _dumpSamples(smp, track, track_index, segs, workspace, num_samples, pattern):
    """--output-samples-pattern: BED with one `track name=<sample>` block per sample of the open sampler `smp`; like
    the reference, every unit's placed list is written under its own key -- `contig` or `contig.isochore` -- before
    fromIsochores (gat/__init__.py:518-559), so the file feeds the same-placement fixture route of the reference."""
    problem = TrackProblem(segs, workspace)
    filename = re.sub("%s", track, pattern)
    dirname = os.path.dirname(filename)
    if dirname and not os.path.exists(dirname):
        os.makedirs(dirname)
    with _open(filename, "w") as outf:
        step = 256
        for b in range(0, num_samples, step):
            placed, _ = smp.place_units(Engine.getSeed(), track_index, b, min(step, num_samples - b))
            for i, per_unit in enumerate(placed):
                outf.write("track name=%i\n" % (b + i))
                for u, arr in enumerate(per_unit):
                    key = problem.unit_keys[u]
                    outf.write("".join("%s\t%i\t%i\n" % (key, s, e) for s, e in arr.tolist()))


def fromCounts(filename):
    """annotator results from a counts table written with output_counts_pattern (gat/__init__.py:1091-1119).  The
    table is parsed on the GPU (Engine.readCountsTable) and the statistics of all rows come from one call; the samples
    stay on the device, as after run().  Tables the GPU reader does not take go through _fromCountsHost."""
    table = Engine.readCountsTable(filename)
    if table is None:
        return _fromCountsHost(filename)
    rows, matrix = table
    st = getContext().column_stats(None, [r[2] for r in rows], pseudo_count=1.0, device_ptr=matrix._tensor.data_ptr(),
                                   n_samples=matrix.nsamples, n_cols=matrix.ncolumns, is_float=0)
    return [AnnotatorResult(track=track, annotation=annotation, counter="na", observed=observed, samples=(matrix, i),
                            stats=dict((k, float(v[i])) for k, v in st.items()))
            for i, (track, annotation, observed) in enumerate(rows)]


def _fromCountsHost(filename):
    """fromCounts parsed on the host, line by line as the reference does"""
    results = []
    with _open(filename, "r") as infile:
        header = infile.readline()
        if not header == "track\tannotation\tobserved\tcounts\n":
            raise ValueError("%s not a counts file: got %s" % (infile, header))
        for line in infile:
            track, annotation, observed, counts = line[:-1].split("\t")
            samples = np.array(list(map(float, counts.split(","))), dtype=np.float64)
            results.append(AnnotatorResult(track=track, annotation=annotation, counter="na",
                                           observed=float(observed), samples=samples))
    return results


from .cli import buildParser  # noqa: E402  (flags of gat.buildParser, gat/__init__.py:54-429)
from .shards import combineShards, mergeShardPrefix, mergeShards  # noqa: E402
