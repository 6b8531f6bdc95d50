"""gat_b200 -- B200-native simulation engine of the Genomic Association Tester.

Drop-in for the `gat.run()` / gat-run.py path of AndreasHeger/gat (gat/__init__.py:855-1088): same
arguments, same result objects, same output table.  The per-sample work of the reference
(UnconditionalSampler.sample -> computeSample, gat/__init__.py:494-591, 704-778) is replaced by batched
CUDA kernels reached through the C ABI in include/gat_b200.h.  One process per GPU; with
torch.distributed initialised the samples are sharded by rank and the count matrix is all-gathered
(gat_b200/parallel.py).
"""
import collections
import re

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


def sampleTrack(track_index, segs, annotations, workspace, sampler, counters, num_samples,
                sample_range=None, annos_cache=None, return_device=False, routes=None):
    """all samples of one track: counts[counter_id] = ndarray [num_samples][n_annot]
    (replaces UnconditionalSampler.sample, gat/__init__.py:704-778).
    routes: output routes (device.Context.set_output_routes) -- the counting kernels deliver the rows straight to
    their consumers (other ranks' matrices included) instead of a local slab."""
    import torch
    ctx = getContext()
    counter_names = [c.name for c in counters]
    atracks = list(annotations.tracks)
    smp, annos = trackSampler(segs, annotations, workspace, sampler, annos_cache)
    if smp is None:
        return atracks, [np.zeros((num_samples, len(atracks))) for _ in counters], np.zeros(3, dtype=np.uint64)
    begin, end = sample_range if sample_range is not None else (0, num_samples)
    n_local = end - begin
    dev = torch.device("cuda", ctx.device)
    ids = device.counter_ids(counter_names)
    # (torch's legacy default stream has handle 0 = "the library's own stream" at the C ABI: pass cudaStreamLegacy)
    ctx.set_stream(torch.cuda.current_stream(dev).cuda_stream or 1)
    if routes is not None:
        out_u = out_f = None
        if n_local > 0:
            ctx.set_output_routes(routes)
            try:
                info = smp.run(annos, counter_names, Engine.getSeed(), track_index, begin, n_local,
                               out_counts_ptr=routes[0]["base"])
            finally:
                ctx.set_output_routes([])
        else:
            info = np.zeros(3, dtype=np.uint64)
    else:
        out_u = torch.zeros((len(ids), max(n_local, 1), len(atracks)), dtype=torch.int32, device=dev)
        out_f = torch.zeros((max(n_local, 1), len(atracks)), dtype=torch.float64, device=dev) \
            if device.DENSITY in ids else None
        info = smp.run(annos, counter_names, Engine.getSeed(), track_index, begin, n_local,
                       out_counts_ptr=out_u.data_ptr(), out_density_ptr=out_f.data_ptr() if out_f is not None else None)
    smp.close()
    if annos_cache is None:
        annos.close()
    return atracks, (out_u, out_f, ids), info


def run(segments, annotations, workspace, sampler, counters, workspace_generator, **kwargs):
    """run an enrichment analysis (signature and kwargs of gat.run, gat/__init__.py:855-907).

    kwargs: num_samples (10000), pseudo_count (1.0), reference, output_counts_pattern,
    output_samples_pattern, outfiles, cache / sample_files / num_threads (accepted, unused: the
    reference's sample cache is dead code and its multiprocessing is replaced by the GPU);
    exchange ("auto" | "allgather" | "columns": how a multi-GPU run combines its slabs, see below);
    keep_samples (None | True | False): False computes the statistics without the sample matrix
    (gat_b200/matrixfree.py), so that the number of samples is not bounded by GPU memory -- the results are the
    same, but their samples cannot be asked for; None (default) does so only when the matrices would not fit in
    the free GPU memory and no counts table is written.
    """
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
            return _run(segments, annotations, workspace, sampler, counters, workspace_generator, **kwargs)
        finally:
            torch.cuda.synchronize(dev)
            ctx.set_stream(None)


def _run(segments, annotations, workspace, sampler, counters, workspace_generator, **kwargs):
    from . import parallel
    import torch

    num_samples = kwargs.get("num_samples", 10000)
    output_counts_pattern = kwargs.get("output_counts_pattern", None)
    output_samples_pattern = kwargs.get("output_samples_pattern", None)
    pseudo_count = kwargs.get("pseudo_count", 1.0)
    reference = kwargs.get("reference", None)

    if not getattr(sampler, "accelerated", False):
        raise NotImplementedError("sampler %s is not accelerated by gat_b200 (only SamplerAnnotator is)"
                                  % type(sampler).__name__)
    if getattr(workspace_generator, "is_conditional", False):
        raise NotImplementedError("conditional workspaces are not accelerated by gat_b200")

    ctx = getContext()
    rank, world = parallel.rank_world()
    import os
    import sys
    import time
    # every rank must place with the SAME seed (the matrix is keyed by seed and global sample index): an
    # unseeded run draws its seed on rank 0 and broadcasts it
    parallel.join_warm_up()
    parallel.share_seed()
    timing = [("start", time.perf_counter())] if os.environ.get("GATB_TIMING") else None

    def mark(name):
        if timing is not None:
            torch.cuda.synchronize(ctx.device)
            timing.append((name, time.perf_counter()))

    # observed counts (gat/__init__.py:932-940)
    annos_cache = {}      # key tuple -> device.Annotations: one upload + index build per key set for the whole run
    observed_counts = [Engine.computeCounts(counter=c, aggregator=sum, segments=segments,
                                            annotations=annotations, workspace=workspace,
                                            workspace_generator=workspace_generator, annos_cache=annos_cache)
                       for c in counters]
    mark("observed")

    # How the per-rank slabs [S/G][A] become statistics (SURVEY 8e / 8f2):
    #   "allgather"  ONE all-gather per counter: every rank holds the S x A matrix (what north_star names)
    #   "columns"    ONE all-to-all per counter: rank g holds all S samples of ITS A/G columns, computes their
    #                statistics, and only the <= 6 x A result doubles are gathered -- 1/G of the traffic and memory
    #   "auto"       columns once the gathered matrices would exceed 1 GiB per rank (and no counts table is wanted:
    #                that needs every column on rank 0)
    exchange = kwargs.get("exchange", os.environ.get("GATB_EXCHANGE", "auto"))
    if exchange not in ("auto", "allgather", "columns"):
        raise ValueError("exchange must be auto, allgather or columns")
    n_atracks = len(list(annotations.tracks))
    if exchange == "auto":
        big = 4 * num_samples * n_atracks * len(counters) >= (1 << 30)
        exchange = "columns" if (world > 1 and big and not output_counts_pattern) else "allgather"
    if world == 1:
        exchange = "allgather"
    if exchange == "columns" and output_counts_pattern:
        raise ValueError("output_counts_pattern needs every column on rank 0: use exchange='allgather'")
    col_begin, col_end = parallel.column_range(n_atracks, rank, world) if exchange == "columns" else (0, n_atracks)

    # keep the S x A matrices, or stream the samples through column accumulators (the exchange and the transport
    # below do not apply then: every rank counts its own samples of all columns, the integers are summed)
    density = any(c.name == "nucleotide-density" for c in counters)
    keep_samples = kwargs.get("keep_samples", None)
    matrix_bytes = 4 * len(counters) * num_samples * (col_end - col_begin) * len(segments.tracks)
    free_bytes = torch.cuda.mem_get_info(ctx.device)[0] if keep_samples is None else 0
    matrix_free = matrixfree.use_matrix_free(keep_samples, bool(output_counts_pattern), density, matrix_bytes, free_bytes)
    if keep_samples is None and world > 1:          # (the free memory differs between GPUs: every rank takes one mode)
        matrix_free = any(matrixfree.allgather(matrix_free, world))

    # Transport of a multi-GPU exchange:
    #   "peer"  the counting kernels store every finished row straight into the destination ranks' matrices (CUDA IPC
    #           memory over NVLink, output routes of the C ABI): the exchange happens inside the kernels' epilogue,
    #           no collective follows; integer counters
    #   "nccl"  the slabs are exchanged with one NCCL collective per counter plane after the kernels
    transport = kwargs.get("transport", os.environ.get("GATB_TRANSPORT", "peer"))
    if transport not in ("peer", "nccl"):
        raise ValueError("transport must be peer or nccl")
    if world == 1 or any(c.name == "nucleotide-density" for c in counters):
        transport = "nccl"              # (one rank: nothing to exchange; the float64 density plane is not routed)

    sampled = {}
    begin, end = parallel.shard_range(num_samples, rank, world)
    streamed = None
    if matrix_free:
        streamed = _sampleStreamed(segments, annotations, workspace, sampler, counters, observed_counts, reference,
                                   num_samples, pseudo_count, annos_cache, rank, world)
        sampled = dict((track, (list(annotations.tracks), None, None, None)) for track in streamed)
        if output_samples_pattern and rank == 0:
            for ntrack, track in enumerate(segments.tracks):
                if track in streamed:
                    _dumpSamples(track, ntrack, segments[track], workspace, sampler, num_samples, output_samples_pattern)
    for ntrack, track in enumerate(segments.tracks if streamed is None else ()):
        segs = segments[track]
        if workspace.sum() == 0:
            continue
        peer = routes = None
        if transport == "peer":
            # every rank's destination matrix, writable by all: [counter][S][all columns | its own columns]
            width = (col_end - col_begin) if exchange == "columns" else n_atracks
            try:
                peer = parallel.PeerMatrix(ctx, len(counters), num_samples, max(width, 1))
            except parallel.PeerUnavailable as e:       # (raised on every rank alike)
                if rank == 0:
                    sys.stderr.write("# gat_b200.run: %s -- using the NCCL transport\n" % e)
                transport = "nccl"
        if transport == "peer":
            routes = []
            for r in range(world):
                cb, ce = parallel.column_range(n_atracks, r, world) if exchange == "columns" else (0, n_atracks)
                _, rows_r, cols_r = peer.shape_of(r)
                if ce > cb:
                    routes.append(dict(base=peer.pointer(r), plane_stride=rows_r * cols_r, row_stride=cols_r, row0=begin,
                                       col_begin=cb, col_end=ce))
        atracks, out, info = sampleTrack(ntrack, segs, annotations, workspace, sampler, counters,
                                         num_samples, sample_range=(begin, end), annos_cache=annos_cache, routes=routes)
        if isinstance(out, list):          # track without any unit
            sampled[track] = (atracks, None, None, None)
            if peer is not None:
                parallel.barrier()
                peer.close()
            continue
        out_u, out_f, ids = out
        mark("sampling")
        if transport == "peer":
            parallel.barrier()              # every rank's kernels have delivered their rows
            out_u = peer.tensor[:, :, :((col_end - col_begin) if exchange == "columns" else n_atracks)].clone()
            parallel.barrier()              # (nobody frees memory a peer still has mapped for writing)
            peer.close()
        elif exchange == "columns":
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
        sampled[track] = (atracks, out_u, out_f, ids)
        if output_samples_pattern and rank == 0:
            _dumpSamples(track, ntrack, segs, workspace, sampler, num_samples, output_samples_pattern)
    mark("exchange")

    # size / overlap columns of AnnotatorResultExtended: once per track and per annotation, the overlap of a
    # track with every annotation in one GPU call (gat/Engine.pyx:1911-1928 does one intersect per result)
    workspace_size = workspace.sum()
    on_device = getattr(annotations, "onDevice", False)
    anno_sizes = annotations.trackSizes() if on_device else \
        dict((a, (annotations[a].counts(), annotations[a].sum())) for a in annotations.tracks)
    track_sizes = {}
    for track in sampled:
        track_sizes[track] = (segments[track].counts(), segments[track].sum(),
                              Engine.overlapColumns(segments[track], annotations, annos_cache))
    for a in annos_cache.values():
        a.close()
    mark("overlap columns")

    # statistics per (counter, track): one batched column-stats call over all annotations
    annotator_results = []
    for counter_id, (counter, observed_count) in enumerate(zip(counters, observed_counts)):
        for track, r in observed_count.items():
            if track not in sampled:
                continue
            atracks, out_u, out_f, ids = sampled[track]
            annos_in_result = [a for a in r.keys()]
            if workspace.sum() == 0:
                continue
            obs = np.array([r[a] for a in atracks], dtype=np.float64)
            ref = None
            if reference:
                ref = np.array([reference[track][a].fold for a in atracks], dtype=np.float64)
            # the S x A matrix stays on the GPU (Engine.SampleMatrix): results copy it to the host only
            # when their samples are asked for.  Column-sharded: this rank's columns [col_begin, col_end)
            matrix = None
            lo, hi = col_begin, col_end
            ref_l = None if ref is None else ref[lo:hi]
            if streamed is not None:
                st = streamed[track][counter_id]
                matrix = Engine.SamplesNotKept(num_samples, len(atracks))
            elif out_u is None:
                host = np.zeros((num_samples, len(atracks)))
                st = ctx.column_stats(host.astype(np.uint32), obs, pseudo_count=pseudo_count, ref_fold=ref)
            elif hi == lo:              # more ranks than columns: nothing to do here
                st = dict((k, np.zeros(0)) for k in ("expected", "stddev", "lower95", "upper95", "fold", "pvalue"))
                matrix = Engine.SampleMatrix(out_f if counter.name == "nucleotide-density" else out_u[counter_id],
                                             counter.name != "nucleotide-density", first_column=lo)
            elif counter.name == "nucleotide-density":
                st = ctx.column_stats(None, obs[lo:hi], pseudo_count=pseudo_count, ref_fold=ref_l,
                                      device_ptr=out_f.data_ptr(), n_samples=num_samples,
                                      n_cols=hi - lo, is_float=1)
                matrix = Engine.SampleMatrix(out_f, False, first_column=lo)
            else:
                plane = out_u[counter_id]
                st = ctx.column_stats(None, obs[lo:hi], pseudo_count=pseudo_count, ref_fold=ref_l,
                                      device_ptr=plane.data_ptr(), n_samples=num_samples,
                                      n_cols=hi - lo, is_float=0)
                matrix = Engine.SampleMatrix(plane, True, first_column=lo)
            if exchange == "columns" and out_u is not None:
                # the result doubles of every rank's columns: one small all-gather
                # (host tensors: a few kB over the gloo side of the process group -- no NCCL set-up for this)
                keys6 = ("expected", "stddev", "lower95", "upper95", "fold", "pvalue")
                mine = torch.from_numpy(np.stack([st[k] for k in keys6]))
                full = parallel.allgather_columns(mine, len(atracks)).numpy()
                st = dict((k, full[i]) for i, k in enumerate(keys6))
            for ai, annotation in enumerate(atracks):
                if annotation not in annos_in_result:
                    continue
                row = dict((k, float(v[ai])) for k, v in st.items())
                annotator_results.append(AnnotatorResultExtended(
                    track=track, annotation=annotation, counter=counter.name, observed=r[annotation],
                    samples=(matrix, ai) if matrix is not None else host[:, ai], track_segments=segments[track],
                    annotation_segments=None if on_device else annotations[annotation], workspace=workspace,
                    reference=reference[track][annotation] if reference else None,
                    pseudo_count=pseudo_count, stats=row,
                    sizes=dict(track_nsegments=track_sizes[track][0], track_size=track_sizes[track][1],
                               annotation_nsegments=anno_sizes[annotation][0],
                               annotation_size=anno_sizes[annotation][1],
                               overlap_nsegments=track_sizes[track][2][annotation][0],
                               overlap_size=track_sizes[track][2][annotation][1],
                               workspace_size=workspace_size)))

    # dump (large) table with counts (gat/__init__.py:1072-1086).  The reference formats every sample with
    # "%i" in a Python loop; here the text of a whole S x A matrix comes from one GPU call (gatb_format_counts)
    if output_counts_pattern and rank == 0:
        for counter in counters:
            filename = re.sub("%s", counter.name, output_counts_pattern)
            texts = {}                    # id(SampleMatrix) -> (text, column offsets)
            with _open(filename, "w") as outfile:
                outfile.write("track\tannotation\tobserved\tcounts\n")
                for o in annotator_results:
                    if o.counter != counter.name:
                        continue
                    lazy = getattr(o, "_lazy", None)
                    if lazy is not None and lazy[0]._as_uint32:
                        if id(lazy[0]) not in texts:
                            texts[id(lazy[0])] = lazy[0].text()
                        text, off = texts[id(lazy[0])]
                        column = text[int(off[lazy[1]]):int(off[lazy[1] + 1])].tobytes().decode("ascii")
                    else:
                        column = ",".join(["%i" % x for x in o.samples])
                    outfile.write("%s\t%s\t%i\t%s\n" % (o.track, o.annotation, o.observed, column))
    torch.cuda.synchronize(ctx.device)
    mark("statistics+results")
    if timing is not None and rank == 0:
        sys.stderr.write("# gat_b200.run phases: " + ", ".join(
            "%s %.3fs" % (timing[i][0], timing[i][1] - timing[i - 1][1]) for i in range(1, len(timing))) + "\n")
    return annotator_results


def _sampleStreamed(segments, annotations, workspace, sampler, counters, observed_counts, reference, num_samples,
                    pseudo_count, annos_cache, rank, world):
    """the matrix-free mode of run(): per track, this rank's samples in slabs of one reused device buffer, counted
    into column accumulators and overwritten; the statistics of the track are complete (summed over the ranks)
    before the next track starts.  -> {track: [statistics dict per counter]}"""
    import torch
    from . import parallel
    ctx = getContext()
    dev = torch.device("cuda", ctx.device)
    names = [c.name for c in counters]
    atracks = list(annotations.tracks)
    A = len(atracks)
    begin, end = parallel.shard_range(num_samples, rank, world)
    n_local = end - begin
    matrixfree.info.update(reruns=0, arena_bytes=0, chunk_rows=0)
    chunk = max(1, min(max(n_local, 1), matrixfree.SLAB_BYTES // (4 * len(names) * max(A, 1))))
    slab = torch.zeros(len(names) * chunk * max(A, 1), dtype=torch.int32, device=dev)
    ctx.set_stream(torch.cuda.current_stream(dev).cuda_stream or 1)
    out = {}
    for ntrack, track in enumerate(segments.tracks):
        if workspace.sum() == 0:
            continue
        smp, annos = trackSampler(segments[track], annotations, workspace, sampler, annos_cache)

        def produce(r0, n):
            if smp is None:                     # a track without any unit: every sample counts zero
                slab[:len(names) * n * A].zero_()
            else:
                smp.run(annos, names, Engine.getSeed(), ntrack, begin + r0, n, out_counts_ptr=slab.data_ptr())
            return slab.data_ptr()

        planes = []
        for counter_id in range(len(counters)):
            r = observed_counts[counter_id][track]
            planes.append((np.array([r[a] for a in atracks], dtype=np.float64),
                           np.array([reference[track][a].fold for a in atracks], dtype=np.float64) if reference else None))
        try:
            out[track] = matrixfree.stream_statistics(ctx, produce, planes, num_samples, n_local, A, chunk,
                                                      pseudo_count=pseudo_count, rank=rank, world=world)
        finally:
            if smp is not None:
                smp.close()
    return out


def _open(filename, mode):
    import gzip
    if filename.endswith(".gz"):
        return gzip.open(filename, mode + "t")
    return open(filename, mode)


def _dumpSamples(track, track_index, segs, workspace, sampler, num_samples, pattern):
    """--output-samples-pattern: BED with one `track name=<sample>` block per sample; like the reference, every
    unit's placed list is written under its own key -- `contig` or `contig.isochore` -- before fromIsochores
    (gat/__init__.py:518-559), so the file feeds the same-placement fixture route of the reference."""
    import os
    ctx = getContext()
    problem = TrackProblem(segs, workspace)
    filename = re.sub("%s", track, pattern)
    dirname = os.path.dirname(filename)
    if dirname and not os.path.exists(dirname):
        os.makedirs(dirname)
    smp = device.Sampler(ctx, problem.unit_contig, len(problem.contigs), problem.has_isochores,
                         problem.unit_segments, problem.unit_workspace,
                         bucket_size=sampler.bucket_size, nbuckets=sampler.nbuckets)
    if getattr(sampler, "kind", "annotator") == "shift":
        smp.set_shift(sampler.radius, sampler.extension)
    elif getattr(sampler, "kind", "annotator") != "annotator":
        smp.set_kind(sampler.kind)
    with _open(filename, "w") as outf:
        step = 256
        for b in range(0, num_samples, step):
            placed, _ = smp.place_units(Engine.getSeed(), track_index, b, min(step, num_samples - b))
            for i, per_unit in enumerate(placed):
                outf.write("track name=%i\n" % (b + i))
                for u, arr in enumerate(per_unit):
                    key = problem.unit_keys[u]
                    outf.write("".join("%s\t%i\t%i\n" % (key, s, e) for s, e in arr.tolist()))
    smp.close()


def fromCounts(filename):
    """annotator results from a counts table written with output_counts_pattern (gat/__init__.py:1091-1119)"""
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
