"""gat/_b200.py -- the binding a maintainer of AndreasHeger/gat would add to route the simulation hot path of the
UNMODIFIED reference through libgat_b200.so (INTEGRATION.md section 2).

It uses nothing but ctypes, numpy and the reference's own containers -- no import of the gat_b200 package -- and is
exercised by tests/test_gpu_dropin.py, which installs it, hands it containers shaped like the reference's and calls
it the way the reference's gat.run() does.

    import gat, _b200
    _b200.install(gat)            # UnconditionalSampler.sample and Engine.computeCounts now call the library
    _b200.seed(1)                 # counterpart of numpy.random.seed(...) in scripts/gat-run.py:267-271
    results = gat.run(segments, annotations, workspace, gat.Engine.SamplerAnnotator(...), counters,
                      gat.Engine.UnconditionalWorkspace(), num_samples=1000)

Replaced reference code: UnconditionalSampler.sample (gat/__init__.py:704-778), i.e. the computeSample loop
(:494-591), and Engine.computeCounts (gat/Engine.pyx:2164-2204).  Everything else of gat.run -- result objects,
statistics, q-values, output -- stays the reference's.
"""
import collections
import ctypes
import os

import numpy

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GATB_LIB") or os.path.join(_HERE, "..", "gat_b200", "lib", "libgat_b200.so")

_vp, _u64, _u32, _i32, _dbl = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int, ctypes.c_double

# GATB_* counter ids of include/gat_b200.h by Counter.name (gat/Engine.pyx:1412-1472)
COUNTER_ID = {"nucleotide-overlap": 0, "nucleotide-density": 1, "segment-overlap": 2, "segment-midoverlap": 3,
              "annotation-overlap": 4, "annotation-midoverlap": 5}
ERR_TOO_LARGE = -4

_lib = None
_ctx = None
_state = {"seed": None, "tracks": {}}


def lib():
    global _lib
    if _lib is None:
        L = ctypes.CDLL(LIB_PATH)
        L.gatb_create.argtypes = [_i32, ctypes.POINTER(_vp)]
        L.gatb_last_error.restype = ctypes.c_char_p
        L.gatb_last_error.argtypes = [_vp]
        L.gatb_destroy.argtypes = [_vp]
        L.gatb_sampler_create.argtypes = [_vp, _i32, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _u32, _u32,
                                          ctypes.POINTER(_vp)]
        L.gatb_sampler_destroy.argtypes = [_vp]
        L.gatb_sampler_set_kind.argtypes = [_vp, _i32]
        L.gatb_sampler_set_shift.argtypes = [_vp, _dbl, _i32]
        L.gatb_annotations_create.argtypes = [_vp, _i32, _i32, _vp, _vp, _vp, _vp, ctypes.POINTER(_vp)]
        L.gatb_annotations_destroy.argtypes = [_vp]
        L.gatb_run.argtypes = [_vp, _vp, _i32, _vp, _u64, _u32, _u64, _u64, _vp, _vp, _i32, _vp]
        L.gatb_count_lists.argtypes = [_vp, _vp, _i32, _vp, _u64, _vp, _vp, _vp, _vp, _vp]
        _lib = L
    return _lib


def context():
    """one library context (GPU LOCAL_RANK or 0) for the process"""
    global _ctx
    if _ctx is None:
        h = _vp()
        rc = lib().gatb_create(int(os.environ.get("LOCAL_RANK", "0")), ctypes.byref(h))
        if rc != 0:
            raise RuntimeError("libgat_b200: %s" % lib().gatb_last_error(None).decode())
        _ctx = h
    return _ctx


def _check(rc):
    if rc == 0:
        return
    msg = lib().gatb_last_error(context()).decode()
    if rc == ERR_TOO_LARGE:
        raise ValueError(msg)                      # getLengthDistribution's error (gat/SegmentList.pyx:1170)
    if rc == -1:
        raise AssertionError(msg)                  # non-normalized input: the reference asserts
    raise RuntimeError("libgat_b200 error %i: %s" % (rc, msg))


def seed(value):
    _state["seed"] = int(value) & 0xFFFFFFFFFFFFFFFF
    _state["tracks"] = {}


def _seed():
    if _state["seed"] is None:                     # an unseeded run draws its seed from numpy's global generator
        seed(int(numpy.random.randint(0, 2 ** 31 - 1)))
    return _state["seed"]


def _p(a):
    return None if a is None else a.ctypes.data_as(_vp)


def _array(sl):
    """reference SegmentList -> (n, 2) uint32 view of its Segment buffer (pickled as raw {uint32 start, end}
    pairs, gat/SegmentList.pyx:314-337)"""
    if len(sl) == 0:
        return numpy.zeros((0, 2), numpy.uint32)
    return numpy.frombuffer(sl.__reduce__()[1][5], dtype=numpy.uint32).reshape(-1, 2)


def _csr(segmentlists):
    arrays = [_array(sl) for sl in segmentlists]
    offs = numpy.zeros(len(arrays) + 1, numpy.uint64)
    if arrays:
        offs[1:] = numpy.cumsum([len(a) for a in arrays])
    data = numpy.concatenate(arrays) if arrays and offs[-1] else numpy.zeros((1, 2), numpy.uint32)
    return offs, numpy.ascontiguousarray(data[:, 0]), numpy.ascontiguousarray(data[:, 1])


def _contig(key):
    key = key.strip()
    return key.split(".")[0] if "." in key and key != "." else key                     # gat/Engine.pyx:2862-2866


def sample_track(track_index, segs, annotations, workspace, sampler, counters, num_samples):
    """body of UnconditionalSampler.sample(): counts_per_track[counter_id][annotation] = list of num_samples"""
    L, ctx = lib(), context()
    contig_annotations = annotations.clone()
    contig_annotations.fromIsochores()                                                  # gat/__init__.py:716-721
    contig_workspace = workspace.clone()
    contig_workspace.fromIsochores()
    keys = [k for k in segs.keys() if not workspace[k].isEmpty and not segs[k].isEmpty]  # :536-538
    tracks = list(annotations.tracks)
    counts = [collections.defaultdict(list) for _ in counters]
    if not keys:
        for ci in range(len(counters)):
            for a in tracks:
                counts[ci][a] = [0] * num_samples
        return counts
    contigs = []
    for k in keys:
        if _contig(k) not in contigs:
            contigs.append(_contig(k))
    unit_contig = numpy.array([contigs.index(_contig(k)) for k in keys], numpy.int32)
    has_iso = int(any(_contig(k) != k.strip() for k in keys))
    so, ss, se = _csr([segs[k] for k in keys])
    wo, ws, we = _csr([workspace[k] for k in keys])
    kind = type(sampler).__name__
    red = sampler.__reduce__()                     # (constructor, (bucket_size, nbuckets, ...) / (radius, extension)):
    if len(red) == 1:                              # the fields are cdef; SamplerShift.__reduce__ nests its tuple once more
        red = red[0]
    args = red[1]
    bucket_size, nbuckets = (1, 0) if kind == "SamplerShift" else (int(args[0]), int(args[1]))
    smp = _vp()
    _check(L.gatb_sampler_create(ctx, len(keys), _p(unit_contig), len(contigs), has_iso, _p(so), _p(ss), _p(se),
                                 _p(wo), _p(ws), _p(we), bucket_size, nbuckets, ctypes.byref(smp)))
    try:
        if kind == "SamplerShift":
            _check(L.gatb_sampler_set_shift(smp, float(args[0]), int(args[1])))
        elif kind == "SamplerSegments":
            _check(L.gatb_sampler_set_kind(smp, 1))
        elif kind != "SamplerAnnotator":
            raise NotImplementedError("sampler %s is not accelerated" % kind)
        empty = type(segs[keys[0]])()
        ao, as_, ae = _csr([contig_annotations[a][c] if c in contig_annotations[a] else empty
                            for a in tracks for c in contigs])
        nseg = numpy.array([len(contig_workspace[c]) for c in contigs], numpy.uint32)
        ann = _vp()
        _check(L.gatb_annotations_create(ctx, len(tracks), len(contigs), _p(ao), _p(as_), _p(ae), _p(nseg),
                                         ctypes.byref(ann)))
        try:
            ids = numpy.array([COUNTER_ID[c.name] for c in counters], numpy.int32)
            out = numpy.zeros((len(ids), num_samples, len(tracks)), numpy.uint32)
            dens = numpy.zeros((num_samples, len(tracks)), numpy.float64)
            info = numpy.zeros(3, numpy.uint64)
            _check(L.gatb_run(smp, ann, len(ids), _p(ids), _seed(), track_index, 0, num_samples, _p(out), _p(dens),
                              0, _p(info)))
        finally:
            L.gatb_annotations_destroy(ann)
    finally:
        L.gatb_sampler_destroy(smp)
    for ci, c in enumerate(counters):
        m = dens if c.name == "nucleotide-density" else out[ci]
        for ai, a in enumerate(tracks):
            counts[ci][a] = m[:, ai].tolist()
    return counts


def compute_counts(counter, aggregator, segments, annotations, workspace, workspace_generator, append=False):
    """Engine.computeCounts (gat/Engine.pyx:2164-2204) for aggregator=sum: one gatb_count_lists call for all
    (track, annotation) pairs, per workspace key with key_ws_nseg = len(workspace[key])"""
    if aggregator is not sum or getattr(workspace_generator, "is_conditional", False):
        raise NotImplementedError("only the unconditional sum of gat.run is bound")
    L, ctx = lib(), context()
    counts = collections.defaultdict(list) if append else collections.defaultdict(lambda: collections.defaultdict(float))
    keys = list(workspace.keys())
    tracks, atracks = list(segments.tracks), list(annotations.tracks)
    if not keys or not tracks or not atracks:
        return counts
    empty = type(workspace[keys[0]])()
    ao, as_, ae = _csr([annotations[a][k] if k in annotations[a] else empty for a in atracks for k in keys])
    nseg = numpy.array([len(workspace[k]) for k in keys], numpy.uint32)
    ann = _vp()
    _check(L.gatb_annotations_create(ctx, len(atracks), len(keys), _p(ao), _p(as_), _p(ae), _p(nseg), ctypes.byref(ann)))
    try:
        so, ss, se = _csr([segments[t][k] if k in segments[t] else empty for t in tracks for k in keys])
        ids = numpy.array([COUNTER_ID[counter.name]], numpy.int32)
        out = numpy.zeros((1, len(tracks), len(atracks)), numpy.float64)
        _check(L.gatb_count_lists(ctx, ann, 1, _p(ids), len(tracks), _p(so), _p(ss), _p(se), None, _p(out)))
    finally:
        L.gatb_annotations_destroy(ann)
    is_float = counter.name == "nucleotide-density"
    for ti, track in enumerate(tracks):
        for ai, annotation in enumerate(atracks):
            v = float(out[0, ti, ai]) if is_float else int(out[0, ti, ai])
            if append:
                counts[annotation].append(v)
            else:
                counts[track][annotation] = v
    return counts


def install(gat):
    """the three-line dispatch of INTEGRATION.md, applied from outside: the reference's own gat.run() now reaches
    the library for the sampling loop and the observed counts.  Returns a function that undoes it."""
    original_sample = gat.UnconditionalSampler.sample
    original_counts = gat.Engine.computeCounts

    def sample(self, track, counts, counters, segs, annotations, workspace, outfiles):
        if getattr(self.workspace_generator, "is_conditional", False):
            return original_sample(self, track, counts, counters, segs, annotations, workspace, outfiles)
        if workspace.sum() == 0:                                                         # gat/__init__.py:733-735
            return None
        index = _state["tracks"].setdefault(track, len(_state["tracks"]))
        return sample_track(index, segs, annotations, workspace, self.sampler, counters, self.num_samples)

    gat.UnconditionalSampler.sample = sample
    gat.Engine.computeCounts = compute_counts

    def uninstall():
        gat.UnconditionalSampler.sample = original_sample
        gat.Engine.computeCounts = original_counts
    return uninstall
