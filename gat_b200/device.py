"""numpy-facing wrappers of the C ABI (include/gat_b200.h): Context, Annotations, Sampler.

Interval lists are numpy arrays of shape (n, 2), dtype uint32, rows [start, end), sorted and
normalized (what SegmentList.normalize() yields in the reference, gat/SegmentList.pyx:697-754).
Everything here only flattens lists to CSR and calls libgat_b200.so; all interval arithmetic of the hot
path runs on the GPU.
"""
import ctypes

import numpy as np

from . import _lib

COUNTERS = ["nucleotide-overlap", "nucleotide-density", "segment-overlap",
            "segment-midoverlap", "annotation-overlap", "annotation-midoverlap",
            "overlap-pieces"]          # the last one is internal (GATB_OVERLAP_PIECES), not a --counter
COUNTER_ID = {name: i for i, name in enumerate(COUNTERS)}
DENSITY = COUNTER_ID["nucleotide-density"]

UNIT_HIT_ROUND_CAP = 1
UNIT_OVERFLOW = 2


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def as_segs(x):
    a = np.asarray(x, dtype=np.uint32).reshape(-1, 2)
    return a


def to_csr(lists):
    """list of (n,2) arrays -> (offs uint64[n+1], start uint32[], end uint32[])"""
    offs = np.zeros(len(lists) + 1, dtype=np.uint64)
    if len(lists):
        offs[1:] = np.cumsum([len(x) for x in lists], dtype=np.uint64)
    total = int(offs[-1])
    if total:
        data = np.concatenate([as_segs(x) for x in lists if len(x)], axis=0)
    else:
        data = np.zeros((0, 2), dtype=np.uint32)
    start = np.ascontiguousarray(data[:, 0])
    end = np.ascontiguousarray(data[:, 1])
    if total == 0:                      # keep valid pointers for ctypes
        start = np.zeros(1, dtype=np.uint32)
        end = np.zeros(1, dtype=np.uint32)
    return offs, start, end


def _host_matrix(counts):
    """a host sample matrix as the statistics entry points take it -> (matrix, is_float, n_samples, n_cols): float64
    stays float64, anything else becomes uint32, both C-contiguous"""
    counts = np.ascontiguousarray(counts)
    is_float = int(counts.dtype == np.float64)
    if not is_float:
        counts = np.ascontiguousarray(counts, dtype=np.uint32)
    n_samples, n_cols = counts.shape
    return counts, is_float, n_samples, n_cols


def counter_ids(counters):
    ids = []
    for c in counters:
        ids.append(COUNTER_ID[c] if isinstance(c, str) else int(c))
    return np.array(ids, dtype=np.int32)


class Context(object):
    """one GPU + one CUDA stream (gatb_ctx)."""

    def __init__(self, device=0):
        self.lib = _lib.load()
        h = ctypes.c_void_p()
        rc = self.lib.gatb_create(int(device), ctypes.byref(h))
        if rc != _lib.OK:
            raise _lib.GatB200Error(rc, self.lib.gatb_last_error(None).decode())
        self.handle = h
        self.device = int(device)

    def check(self, rc):
        if rc != _lib.OK:
            raise _lib.GatB200Error(rc, self.lib.gatb_last_error(self.handle).decode())

    def close(self):
        if getattr(self, "handle", None):
            self.lib.gatb_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream_ptr):
        self.check(self.lib.gatb_set_stream(self.handle, ctypes.c_void_p(cuda_stream_ptr or 0)))

    def synchronize(self):
        self.check(self.lib.gatb_synchronize(self.handle))

    def set_batch_size(self, batch):
        self.check(self.lib.gatb_set_batch_size(self.handle, int(batch)))

    @property
    def launch_count(self):
        return int(self.lib.gatb_launch_count(self.handle))

    def profile(self, enable=True):
        """bracket every kernel launch with CUDA events (see profile_read)"""
        self.check(self.lib.gatb_profile(self.handle, int(bool(enable))))

    def profile_read(self):
        """-> {class: (device ms, launches)} accumulated since the last read; classes place/merge/count/other"""
        ms = np.zeros(4, dtype=np.float64)
        n = np.zeros(4, dtype=np.uint64)
        self.check(self.lib.gatb_profile_read(self.handle, _p(ms), _p(n)))
        return dict((k, (float(ms[i]), int(n[i]))) for i, k in enumerate(["place", "merge", "count", "other"]))

    def column_stats(self, counts, observed, pseudo_count=1.0, ref_fold=None, device_ptr=None,
                     n_samples=None, n_cols=None, is_float=None):
        """per-column expected/stddev/CI95/fold/pvalue (gat/Engine.pyx:1635-1718).

        counts: host ndarray [n_samples][n_cols] uint32 or float64; or pass device_ptr (+ shape)."""
        if device_ptr is None:
            counts, is_float, n_samples, n_cols = _host_matrix(counts)
            ptr, on_dev = _p(counts), 0
        else:
            ptr, on_dev = ctypes.c_void_p(device_ptr), 1
        obs = np.ascontiguousarray(observed, dtype=np.float64)
        ref = None if ref_fold is None else np.ascontiguousarray(ref_fold, dtype=np.float64)
        outs = [np.zeros(n_cols, dtype=np.float64) for _ in range(6)]
        self.check(self.lib.gatb_column_stats(self.handle, ptr, int(is_float), on_dev, int(n_samples), int(n_cols),
                                              _p(obs), _p(ref), float(pseudo_count), *[_p(o) for o in outs]))
        return dict(zip(["expected", "stddev", "lower95", "upper95", "fold", "pvalue"], outs))


    def set_output_routes(self, routes):
        """routes: list of dicts(base=device pointer, plane_stride, row_stride, row0, col_begin, col_end) -- where the
        counting kernels of the following gatb_run calls deliver their integer results (gatb_set_output_routes);
        an empty list restores the plain output"""
        arr = (_lib.Route * max(len(routes), 1))()
        for i, r in enumerate(routes):
            arr[i] = _lib.Route(int(r["base"]), int(r.get("plane_stride", 0)), int(r["row_stride"]), int(r.get("row0", 0)),
                                int(r["col_begin"]), int(r["col_end"]))
        self.check(self.lib.gatb_set_output_routes(self.handle, len(routes), ctypes.byref(arr)))

    def set_route_mode(self, by_kernel):
        """False (default): copy engines scatter a staging slab to the routes; True: the kernel's epilogue stores to them"""
        self.check(self.lib.gatb_set_route_mode(self.handle, int(bool(by_kernel))))

    def peer_alloc(self, nbytes):
        """shareable device memory -> (pointer, 64-byte IPC handle)"""
        ptr = ctypes.c_void_p()
        handle = (ctypes.c_ubyte * 64)()
        self.check(self.lib.gatb_peer_alloc(self.handle, int(nbytes), ctypes.byref(ptr), ctypes.byref(handle)))
        return int(ptr.value), bytes(handle)

    def peer_free(self, ptr):
        self.check(self.lib.gatb_peer_free(self.handle, ctypes.c_void_p(ptr)))

    def peer_open(self, handle):
        ptr = ctypes.c_void_p()
        buf = (ctypes.c_ubyte * 64).from_buffer_copy(handle)
        self.check(self.lib.gatb_peer_open(self.handle, ctypes.byref(buf), ctypes.byref(ptr)))
        return int(ptr.value)

    def peer_close(self, ptr):
        self.check(self.lib.gatb_peer_close(self.handle, ctypes.c_void_p(ptr)))

    def column_pvalue(self, counts, values, expected):
        """AnnotatorResult.getEmpiricalPValue (gat/Engine.pyx:1829-1831): p-value of values[a] among the samples
        of column a against the STORED expectation expected[a]; counts: host ndarray [n_samples][n_cols]"""
        counts, is_float, n_samples, n_cols = _host_matrix(counts)
        v = np.ascontiguousarray(values, dtype=np.float64)
        e = np.ascontiguousarray(expected, dtype=np.float64)
        out = np.zeros(n_cols, dtype=np.float64)
        self.check(self.lib.gatb_column_pvalue(self.handle, _p(counts), is_float, 0, int(n_samples), int(n_cols),
                                               _p(v), _p(e), _p(out)))
        return out

    def format_counts(self, counts=None, device_ptr=None, n_samples=None, n_cols=None):
        """the text of the counts table (gat/__init__.py:1072-1086): -> (text uint8[], col_off uint64[n_cols+1]);
        column a of the [n_samples][n_cols] uint32 matrix is text[col_off[a]:col_off[a+1]] = b"c0,c1,..."."""
        if device_ptr is None:
            counts = np.ascontiguousarray(counts, dtype=np.uint32)
            n_samples, n_cols = counts.shape
            ptr, on_dev = _p(counts), 0
        else:
            ptr, on_dev = ctypes.c_void_p(device_ptr), 1
        off = np.zeros(n_cols + 1, dtype=np.uint64)
        self.check(self.lib.gatb_format_counts(self.handle, ptr, on_dev, int(n_samples), int(n_cols), _p(off), None, 0))
        text = np.empty(max(int(off[-1]), 1), dtype=np.uint8)
        self.check(self.lib.gatb_format_counts(self.handle, ptr, on_dev, int(n_samples), int(n_cols), _p(off),
                                               _p(text), int(text.size)))
        return text[:int(off[-1])], off

    def compare_stats(self, m1, m2, col1, col2, obs1, obs2, delta, pseudo_count=1.0):
        """gat-compare's pairwise statistics (scripts/gat-compare.py:218-241, :300-323) for pairs
        (column col1[q] of m1, column col2[q] of m2); m1, m2: [n_samples][n_cols] float64 sample matrices"""
        m1 = np.ascontiguousarray(m1, dtype=np.float64)
        m2 = m1 if m2 is None else np.ascontiguousarray(m2, dtype=np.float64)
        if m1.shape[0] != m2.shape[0]:
            raise ValueError("sample matrices differ in the number of samples")
        c1 = np.ascontiguousarray(col1, dtype=np.int32)
        c2 = np.ascontiguousarray(col2, dtype=np.int32)
        arrs = [np.ascontiguousarray(x, dtype=np.float64) for x in (obs1, obs2, delta)]
        n = len(c1)
        outs = [np.zeros(n, dtype=np.float64) for _ in range(6)]
        self.check(self.lib.gatb_compare_stats(self.handle, int(m1.shape[0]), _p(m1), int(m1.shape[1]), _p(m2),
                                               int(m2.shape[1]), n, _p(c1), _p(c2), *[_p(a) for a in arrs],
                                               float(pseudo_count), *[_p(o) for o in outs]))
        return dict(zip(["expected", "stddev", "lower95", "upper95", "fold", "pvalue"], outs))


class ColumnAccumulator(object):
    """the statistics of one uint32 counter plane [n_samples][n_cols] from slabs of rows, without the matrix
    (gatb_colacc): exact sums per column, and unit-width histogram windows for the two CI95 order statistics."""

    STATS = ["expected", "stddev", "lower95", "upper95", "fold", "pvalue"]

    def __init__(self, ctx, n_cols, n_samples, observed, ref_fold=None):
        self.ctx = ctx
        self.n_cols, self.n_samples = int(n_cols), int(n_samples)
        obs = np.ascontiguousarray(observed, dtype=np.float64)
        ref = None if ref_fold is None else np.ascontiguousarray(ref_fold, dtype=np.float64)
        h = ctypes.c_void_p()
        ctx.check(ctx.lib.gatb_colacc_create(ctx.handle, self.n_cols, self.n_samples, _p(obs), _p(ref), ctypes.byref(h)))
        self.handle = h
        self.n_bins = 0

    def set_windows(self, lo, width):
        """column a counts the values lo[a] .. lo[a] + width[a] - 1 into bins; clears the histograms"""
        lo = np.ascontiguousarray(lo, dtype=np.uint32)
        width = np.ascontiguousarray(width, dtype=np.uint32)
        self.ctx.check(self.ctx.lib.gatb_colacc_set_windows(self.handle, _p(lo), _p(width)))
        self.n_bins = int(width.astype(np.uint64).sum())

    def add(self, device_ptr, n_rows, row_stride=None, sums=True, hist=True):
        """count a device slab of n_rows rows (enqueued on the context's stream)"""
        what = (_lib.COLACC_SUMS if sums else 0) | (_lib.COLACC_HIST if hist else 0)
        self.ctx.check(self.ctx.lib.gatb_colacc_add(self.handle, ctypes.c_void_p(device_ptr), int(n_rows),
                                                    int(row_stride or self.n_cols), what))

    def state(self):
        """-> dict of the integer state (rows, moments [5][A], minmax [2][A], outside [2][A], bins)"""
        A = self.n_cols
        rows = np.zeros(1, dtype=np.uint64)
        st = dict(moments=np.zeros((5, A), dtype=np.uint64), minmax=np.zeros((2, A), dtype=np.uint32),
                  outside=np.zeros((2, A), dtype=np.uint64), bins=np.zeros(max(self.n_bins, 1), dtype=np.uint32))
        self.ctx.check(self.ctx.lib.gatb_colacc_state(self.handle, _p(rows), _p(st["moments"]), _p(st["minmax"]),
                                                      _p(st["outside"]), _p(st["bins"])))
        st["rows"] = int(rows[0])
        return st

    def merge(self, st, sums=True):
        """add another accumulator's state (sums=False: only its histograms) into this one"""
        self.ctx.check(self.ctx.lib.gatb_colacc_merge(
            self.handle, st["rows"] if sums else 0, _p(st["moments"]) if sums else None,
            _p(st["minmax"]) if sums else None, _p(st["outside"]), _p(st["bins"])))

    def finish(self, pseudo_count=1.0):
        """-> (statistics dict as Context.column_stats returns it, missed bool [A])"""
        outs = [np.zeros(self.n_cols, dtype=np.float64) for _ in self.STATS]
        missed = np.zeros(self.n_cols, dtype=np.uint8)
        self.ctx.check(self.ctx.lib.gatb_colacc_finish(self.handle, float(pseudo_count), *[_p(o) for o in outs],
                                                       _p(missed)))
        return dict(zip(self.STATS, outs)), missed.astype(bool)

    def close(self):
        if getattr(self, "handle", None):
            if self.ctx.handle:
                self.ctx.lib.gatb_colacc_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Lists(object):
    """interval lists resident on the GPU as CSR (gatb_lists): the device side of input preparation."""

    def __init__(self, ctx, handle):
        self.ctx = ctx
        self.handle = handle
        n_lists, n = ctypes.c_uint32(), ctypes.c_uint64()
        ctx.check(ctx.lib.gatb_lists_info(handle, ctypes.byref(n_lists), ctypes.byref(n)))
        self.n_lists, self.n_intervals = int(n_lists.value), int(n.value)

    @classmethod
    def from_rows(cls, ctx, list_id, start, end, n_lists, join_adjacent=False):
        """rows in any order -> sorted, normalized (join_adjacent: merge(0)-ed) lists"""
        l = np.ascontiguousarray(list_id, dtype=np.uint32)
        s = np.ascontiguousarray(start, dtype=np.uint32)
        e = np.ascontiguousarray(end, dtype=np.uint32)
        h = ctypes.c_void_p()
        ctx.check(ctx.lib.gatb_lists_from_rows(ctx.handle, len(l), _p(l), _p(s), _p(e), int(n_lists),
                                               int(bool(join_adjacent)), ctypes.byref(h)))
        return cls(ctx, h)

    @classmethod
    def from_lists(cls, ctx, lists):
        """normalized host lists ((n,2) arrays) -> device lists"""
        offs, start, end = to_csr(lists)
        h = ctypes.c_void_p()
        ctx.check(ctx.lib.gatb_lists_from_csr(ctx.handle, len(lists), _p(offs), _p(start), _p(end), ctypes.byref(h)))
        return cls(ctx, h)

    def _new(self, fn, *args):
        h = ctypes.c_void_p()
        self.ctx.check(fn(self.handle, *args, ctypes.byref(h)))
        return Lists(self.ctx, h)

    def restrict(self, n_keys, fanout, other, truncate):
        """list l against other[(l % n_keys) * fanout + f] for every f: intersect (truncate) or filter"""
        return self._new(self.ctx.lib.gatb_lists_restrict, int(n_keys), int(fanout), other.handle, int(bool(truncate)))

    def collapse(self, fanout):
        """every `fanout` consecutive lists -> one, merge(0)-ed (fromIsochores)"""
        return self._new(self.ctx.lib.gatb_lists_collapse, int(fanout))

    def select(self, src):
        """out[l] = self[src[l]]; an index >= n_lists gives an empty list"""
        src = np.ascontiguousarray(src, dtype=np.uint32)
        return self._new(self.ctx.lib.gatb_lists_select, len(src), _p(src))

    def sizes(self):
        """-> (len, sum) of every list as uint64 arrays"""
        count = np.zeros(max(self.n_lists, 1), dtype=np.uint64)
        bases = np.zeros(max(self.n_lists, 1), dtype=np.uint64)
        self.ctx.check(self.ctx.lib.gatb_lists_sizes(self.handle, _p(count), _p(bases)))
        return count[:self.n_lists], bases[:self.n_lists]

    def download(self):
        """-> (offs uint64[n_lists + 1], intervals (n, 2) uint32)"""
        offs = np.zeros(self.n_lists + 1, dtype=np.uint64)
        start = np.zeros(max(self.n_intervals, 1), dtype=np.uint32)
        end = np.zeros(max(self.n_intervals, 1), dtype=np.uint32)
        self.ctx.check(self.ctx.lib.gatb_lists_download(self.handle, _p(offs), _p(start), _p(end)))
        return offs, np.stack([start[:self.n_intervals], end[:self.n_intervals]], axis=1)

    def close(self):
        if getattr(self, "handle", None):
            if self.ctx.handle:
                self.ctx.lib.gatb_lists_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Annotations(object):
    """annotation tracks staged on the GPU for counting (gatb_annotations).

    lists[a][k]: intervals of track a on key k (n_annot x n_keys)."""

    @classmethod
    def from_device_lists(cls, ctx, lists, n_annot, n_keys, key_ws_nseg=None):
        """annotation set straight from n_annot x n_keys device lists (no host round trip of the intervals)"""
        self = cls.__new__(cls)
        self.ctx = ctx
        self.n_annot, self.n_keys = int(n_annot), int(n_keys)
        nseg = None if key_ws_nseg is None else np.ascontiguousarray(key_ws_nseg, dtype=np.uint32)
        h = ctypes.c_void_p()
        ctx.check(ctx.lib.gatb_annotations_create_from_lists(ctx.handle, lists.handle, self.n_annot, self.n_keys, _p(nseg),
                                                             ctypes.byref(h)))
        self.handle = h
        self.n_intervals = lists.n_intervals
        self._pending = None
        return self

    def __init__(self, ctx, lists, key_ws_nseg=None, csr=None, lazy=False):
        """lists[a][k], or csr=(n_annot, n_keys, offs, start, end) already flattened annotation-major.

        lazy: gatb_annotations_create_async -- upload and index build run on the library's upload stream
        while the caller goes on (e.g. to the placement kernel); the first run / count_lists waits on the
        device and reports invalid lists.  The arrays are kept alive here until then."""
        self.ctx = ctx
        if csr is not None:
            self.n_annot, self.n_keys, offs, start, end = csr
        else:
            self.n_annot = len(lists)
            self.n_keys = len(lists[0]) if self.n_annot else 0
            flat = [lists[a][k] for a in range(self.n_annot) for k in range(self.n_keys)]
            offs, start, end = to_csr(flat)
        nseg = None if key_ws_nseg is None else np.ascontiguousarray(key_ws_nseg, dtype=np.uint32)
        h = ctypes.c_void_p()
        create = ctx.lib.gatb_annotations_create_async if lazy else ctx.lib.gatb_annotations_create
        ctx.check(create(ctx.handle, self.n_annot, self.n_keys, _p(offs), _p(start), _p(end), _p(nseg),
                         ctypes.byref(h)))
        self.handle = h
        self.n_intervals = int(offs[-1])
        self._pending = (offs, start, end, nseg) if lazy else None

    def wait(self):
        """block until an asynchronous build has finished; raises if the lists were invalid"""
        self.ctx.check(self.ctx.lib.gatb_annotations_wait(self.handle))
        self._pending = None

    def close(self):
        if getattr(self, "handle", None):
            if self.ctx.handle:                                          # (a closed context took its objects along)
                self.ctx.lib.gatb_annotations_destroy(self.handle)       # waits for a pending build
            self.handle = None
            self._pending = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def count_lists(self, counters, samples, key_present=None):
        """samples[s][k]: segment list of sample s on key k -> float64 [n_counters][n_samples][n_annot]"""
        ids = counter_ids(counters)
        n_samples = len(samples)
        flat = [samples[s][k] for s in range(n_samples) for k in range(self.n_keys)]
        offs, start, end = to_csr(flat)
        present = None if key_present is None else np.ascontiguousarray(key_present, dtype=np.uint8)
        out = np.zeros((len(ids), n_samples, self.n_annot), dtype=np.float64)
        self.ctx.check(self.ctx.lib.gatb_count_lists(self.ctx.handle, self.handle, len(ids), _p(ids), n_samples,
                                                     _p(offs), _p(start), _p(end), _p(present), _p(out)))
        return out


class Sampler(object):
    """one segment track + workspace staged on the GPU for placement (gatb_sampler)."""

    def __init__(self, ctx, unit_contig, n_contigs, has_isochores, unit_segments, unit_workspace,
                 bucket_size=1, nbuckets=100000, csr=None):
        """unit_segments / unit_workspace: lists of (n,2) arrays per unit, or csr=(seg_csr, ws_csr) with
        each (offs, start, end) already flattened"""
        self.ctx = ctx
        self.n_units = len(unit_contig)
        self.n_contigs = int(n_contigs)
        uc = np.ascontiguousarray(unit_contig, dtype=np.int32)
        if csr is not None:
            (soffs, sstart, send), (woffs, wstart, wend) = csr
        else:
            soffs, sstart, send = to_csr(unit_segments)
            woffs, wstart, wend = to_csr(unit_workspace)
        h = ctypes.c_void_p()
        ctx.check(ctx.lib.gatb_sampler_create(ctx.handle, self.n_units, _p(uc), self.n_contigs, int(bool(has_isochores)),
                                              _p(soffs), _p(sstart), _p(send), _p(woffs), _p(wstart), _p(wend),
                                              int(bucket_size), int(nbuckets), ctypes.byref(h)))
        self.handle = h
        self.capacity = int(ctx.lib.gatb_sampler_sample_capacity(h))

    def close(self):
        if getattr(self, "handle", None):
            if self.ctx.handle:
                self.ctx.lib.gatb_sampler_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_kind(self, kind):
        """'annotator' (default) or 'segments' (SamplerSegments, isochore workspaces only)"""
        k = {"annotator": 0, "segments": 1}[kind] if isinstance(kind, str) else int(kind)
        self.ctx.check(self.ctx.lib.gatb_sampler_set_kind(self.handle, k))

    def set_shift(self, radius=2, extension=0):
        """SamplerShift(radius, extension) (gat/Engine.pyx:998-1111); re-sizes the sample buffers"""
        self.ctx.check(self.ctx.lib.gatb_sampler_set_shift(self.handle, float(radius), int(extension)))
        self.capacity = int(self.ctx.lib.gatb_sampler_sample_capacity(self.handle))

    def _place(self, by_unit, seed, track, sample_begin, n_samples):
        lib = self.ctx.lib
        fn = lib.gatb_sampler_place_units if by_unit else lib.gatb_sampler_place
        capfn = lib.gatb_sampler_unit_capacity if by_unit else lib.gatb_sampler_sample_capacity
        n_lists = self.n_units if by_unit else self.n_contigs
        while True:
            cap = int(capfn(self.handle))
            start = np.zeros(max(n_samples * cap, 1), dtype=np.uint32)
            end = np.zeros(max(n_samples * cap, 1), dtype=np.uint32)
            counts = np.zeros(max(n_samples * n_lists, 1), dtype=np.uint32)
            base = np.zeros(n_lists, dtype=np.uint64)
            status = np.zeros(max(n_samples * self.n_units, 1), dtype=np.uint8)
            rc = fn(self.handle, int(seed), int(track), int(sample_begin), int(n_samples), _p(start), _p(end),
                    _p(counts), _p(base), _p(status))
            # a unit outgrew its buffer: the library enlarged it; repeat with arrays of the new capacity
            if rc == _lib.ERR_CAPACITY and int(capfn(self.handle)) > cap:
                continue
            self.ctx.check(rc)
            break
        self.capacity = int(lib.gatb_sampler_sample_capacity(self.handle))
        out = []
        for s in range(n_samples):
            per = []
            for c in range(n_lists):
                n = int(counts[s * n_lists + c])
                o = s * cap + int(base[c])
                per.append(np.stack([start[o:o + n], end[o:o + n]], axis=1))
            out.append(per)
        return out, status[:n_samples * self.n_units].reshape(n_samples, self.n_units)

    def place(self, seed, track, sample_begin, n_samples):
        """-> (samples, status): samples[s][c] = (n,2) uint32 array of contig c; status [n_samples][n_units]"""
        return self._place(False, seed, track, sample_begin, n_samples)

    def place_units(self, seed, track, sample_begin, n_samples):
        """-> (samples, status): samples[s][u] = (n,2) uint32 array of UNIT u (key of the track), i.e. what
        sampler.sample(segs[key], workspace[key]) returns before fromIsochores (gat/__init__.py:531-546)"""
        return self._place(True, seed, track, sample_begin, n_samples)

    def run(self, annotations, counters, seed, track, sample_begin, n_samples,
            out_counts_ptr=None, out_density_ptr=None):
        """place + count.  Host mode (default) returns {counter_name: ndarray [n_samples][n_annot]} and info;
        device mode writes into the given device pointers ([n_counters][n_samples][n_annot] uint32 /
        [n_samples][n_annot] float64) and returns only info."""
        ids = counter_ids(counters)
        A = annotations.n_annot
        info = np.zeros(3, dtype=np.uint64)
        if out_counts_ptr is not None or out_density_ptr is not None:
            self.ctx.check(self.ctx.lib.gatb_run(self.handle, annotations.handle, len(ids), _p(ids), int(seed),
                                                 int(track), int(sample_begin), int(n_samples),
                                                 ctypes.c_void_p(out_counts_ptr or 0),
                                                 ctypes.c_void_p(out_density_ptr or 0), 1, _p(info)))
            return info
        out = np.zeros((len(ids), n_samples, A), dtype=np.uint32)
        dens = np.zeros((n_samples, A), dtype=np.float64) if DENSITY in ids else None
        self.ctx.check(self.ctx.lib.gatb_run(self.handle, annotations.handle, len(ids), _p(ids), int(seed),
                                             int(track), int(sample_begin), int(n_samples), _p(out), _p(dens),
                                             0, _p(info)))
        res = {}
        for i, cid in enumerate(ids):
            res[COUNTERS[cid]] = dens if cid == DENSITY else out[i]
        return res, info
