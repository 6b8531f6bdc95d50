"""Statistics of gat_b200.run() without the sample matrix (run(..., keep_samples=False)).

The matrix path holds every sampled count, [S][A] uint32 per (segment track, counter), until the statistics are
computed, so GPU memory bounds the number of samples.  Here the samples of a track are produced in slabs of rows
that are counted and then overwritten: exact integer sums per column (the streamed pass 1 of the column
statistics, accumulating) and, for the two CI95 order statistics, a window of unit-width bins per column around
where a pilot slab puts them (device.ColumnAccumulator, gatb_colacc_* in include/gat_b200.h).  A column whose
rank falls outside its window is counted again over [min, max] of the column: every sample is a function of
(seed, track, unit, global sample index), so the second pass sees the same values.  The results are the
matrix path's, bit for bit; the device memory is one slab plus the windows, whatever S is.
"""
import time

import numpy as np

from . import device

SLAB_BYTES = 512 << 20          # one slab of [counters][rows][columns] uint32
ARENA_FRACTION = 0.25           # histogram windows of one track may take this share of the free device memory
PILOT_WINDOW = None             # (tests) every pilot window this many bins wide, to force the second pass

# what the last matrix-free run did (per process): second sampling passes, largest arena of one track, rows per slab,
# seconds of the shard jobs' histogram passes
info = dict(reruns=0, arena_bytes=0, chunk_rows=0, pass2_seconds=0.0)


def use_matrix_free(keep_samples, counts_table, density, matrix_bytes, free_bytes):
    """run(keep_samples=...) -> True for the matrix-free mode.  keep_samples=True / False is obeyed (False cannot
    write a counts table, and has no float64 density plane); None takes the matrix-free mode only when neither is
    asked for and the matrices the run would hold on this rank do not fit in the free device memory."""
    if keep_samples is None:
        return not counts_table and not density and matrix_bytes > free_bytes
    if not keep_samples:
        if counts_table:
            raise ValueError("output_counts_pattern writes every sample: it needs keep_samples=True")
        if density:
            raise NotImplementedError("nucleotide-density has no matrix-free mode (float64 samples): use keep_samples=True")
        return True
    return False


def pilot_windows(lower, upper):
    """(lo, hi) bounds of the histogram windows from a pilot slab's CI95 bounds: widened by half the interval on
    each side and at least 8 values"""
    lower = np.asarray(lower, dtype=np.float64)
    upper = np.asarray(upper, dtype=np.float64)
    margin = np.maximum(8.0, np.ceil(0.5 * (upper - lower)))
    lo = np.maximum(0.0, np.floor(lower) - margin)
    hi = np.minimum(4294967295.0, np.ceil(upper) + margin)
    return lo.astype(np.int64), hi.astype(np.int64)


def allgather(obj, world):
    if world == 1:
        return [obj]
    import torch.distributed as dist
    box = [None] * world
    dist.all_gather_object(box, obj)
    return box


def _merge_ranks(accs, world, rank, sums):
    """every rank adds the other ranks' integer state into its accumulators (the 128-bit sum of squares with its
    carry, which an element-wise all-reduce of the two words would lose)"""
    if world == 1:
        return
    states = allgather([a.state() for a in accs], world)
    for r, st in enumerate(states):
        if r != rank:
            for a, s in zip(accs, st):
                a.merge(s, sums=sums)


def _slabs(produce, start, n_local, chunk):
    for r0 in range(start, n_local, chunk):
        n = min(chunk, n_local - r0)
        yield n, produce(r0, n)


def _count(accs, n, ptr, n_cols, sums, hist):
    """slab [planes][n][n_cols] at ptr into the accumulators of the planes"""
    for i, a in enumerate(accs):
        a.add(ptr + 4 * i * n * n_cols, n, n_cols, sums=sums, hist=hist)


def _set_windows(accs, lo, hi, budget_bytes, what):
    width = [np.where(h >= l, h - l + 1, 0).astype(np.uint64) for l, h in zip(lo, hi)]
    arena = 4 * int(sum(int(w.sum()) for w in width))
    if arena > budget_bytes:
        raise MemoryError("matrix-free statistics: the %s windows need %i bytes of histogram bins, more than the "
                          "%i bytes allowed (%i columns)" % (what, arena, budget_bytes, int(sum(len(w) for w in width))))
    for a, l, w in zip(accs, lo, width):
        a.set_windows(np.maximum(l, 0).astype(np.uint32), w.astype(np.uint32))
    info["arena_bytes"] = max(info["arena_bytes"], arena)


def stream_statistics(ctx, produce, planes, n_samples, n_local, n_cols, chunk, pseudo_count=1.0,
                      budget_bytes=None, rank=0, world=1):
    """statistics of n_cols columns of len(planes) uint32 counter planes whose n_samples rows are produced in slabs.

    produce(row0, n): rows row0 .. row0 + n - 1 of THIS rank's n_local rows -> device pointer of [planes][n][n_cols]
    uint32, valid until the next call (work on the context's stream is ordered after the counting of the slab).
    planes: [(observed, ref_fold or None)] per plane.  -> [statistics dict per plane], as Context.column_stats."""
    if budget_bytes is None:
        import torch
        budget_bytes = int(ARENA_FRACTION * torch.cuda.mem_get_info(ctx.device)[0])
    accs = [device.ColumnAccumulator(ctx, n_cols, n_samples, obs, ref) for obs, ref in planes]
    try:
        return _stream(ctx, accs, produce, n_local, n_cols, chunk, pseudo_count, budget_bytes, rank, world)
    finally:
        for a in accs:
            a.close()


def _stream(ctx, accs, produce, n_local, n_cols, chunk, pseudo_count, budget_bytes, rank, world):
    P = len(accs)
    chunk = max(1, min(chunk, n_local)) if n_local else 1
    info["chunk_rows"] = chunk

    # pilot: the first slab of this rank; every rank takes the union of all ranks' windows
    lo = [np.full(n_cols, np.iinfo(np.int64).max, dtype=np.int64) for _ in range(P)]
    hi = [np.full(n_cols, -1, dtype=np.int64) for _ in range(P)]
    n0 = min(chunk, n_local)
    ptr0 = produce(0, n0) if n0 else None
    if n0:
        for i in range(P):
            st = ctx.column_stats(None, np.zeros(n_cols), device_ptr=ptr0 + 4 * i * n0 * n_cols, n_samples=n0,
                                  n_cols=n_cols, is_float=0)
            lo[i], hi[i] = pilot_windows(st["lower95"], st["upper95"])
            if PILOT_WINDOW is not None:
                hi[i] = lo[i] + PILOT_WINDOW - 1
    for other in allgather((lo, hi), world):
        for i in range(P):
            lo[i] = np.minimum(lo[i], other[0][i])
            hi[i] = np.maximum(hi[i], other[1][i])
    _set_windows(accs, lo, hi, budget_bytes, "pilot")

    if n0:
        _count(accs, n0, ptr0, n_cols, True, True)
    for n, ptr in _slabs(produce, n0, n_local, chunk):
        _count(accs, n, ptr, n_cols, True, True)
    _merge_ranks(accs, world, rank, sums=True)
    results = [a.finish(pseudo_count) for a in accs]
    if not any(m.any() for _, m in results):
        return [st for st, _ in results]

    # second pass for the columns whose CI rank fell outside the pilot window: [min, max] of the column holds it
    info["reruns"] += 1
    lo2, hi2 = [], []
    for a, (_, m) in zip(accs, results):
        minmax = a.state()["minmax"].astype(np.int64)
        lo2.append(np.where(m, minmax[0], 0))
        hi2.append(np.where(m, minmax[1], -1))
    _set_windows(accs, lo2, hi2, budget_bytes, "second-pass")
    for n, ptr in _slabs(produce, 0, n_local, chunk):
        _count(accs, n, ptr, n_cols, False, True)
    _merge_ranks(accs, world, rank, sums=False)
    out = []
    for a, (st, m) in zip(accs, results):
        st2, m2 = a.finish(pseudo_count)
        if (m & m2).any():
            raise RuntimeError("matrix-free statistics: a CI rank missed the [min, max] window of its column")
        for k in ("lower95", "upper95"):
            st[k] = np.where(m, st2[k], st[k])
        out.append(st)
    return out


# ------------------------------------------------------------------------------------------------ shards
# A shard job (gat_b200.runShard) counts a range of the global samples and keeps the exact integers instead of the
# statistics: the sums of the range and the histogram of every column over the column's whole [min, max] in the
# range.  Integers add across any split of the samples, and a histogram over [min, max] holds every rank, so shards
# of the same run merge into its statistics bit for bit, without sampling again and without agreeing on windows.

def shard_states(ctx, produce, planes, n_samples, n_local, n_cols, chunk, budget_bytes=None, rank=0, world=1):
    """the integer state of this shard's rows of all ranks, for len(planes) uint32 counter planes whose rows are
    produced in slabs (produce, planes, chunk as in stream_statistics).  Pass 1 counts the sums; pass 2 counts the
    histograms over the [min, max] of every column, from the slab still in the buffer when the rank's rows fit in
    one slab, else sampled again.  -> [dict(rows, moments [5][A], minmax [2][A], col_ptr int64 [A+1], value uint32,
    count uint64) per plane]: the gatb_colacc_state layout, the histogram as sparse CSR per column, compacted on the
    device (ColumnAccumulator.export; the layout of sparse_histogram)."""
    if budget_bytes is None:
        import torch
        budget_bytes = int(ARENA_FRACTION * torch.cuda.mem_get_info(ctx.device)[0])
    accs = [device.ColumnAccumulator(ctx, n_cols, n_samples, obs, ref) for obs, ref in planes]
    try:
        chunk = max(1, min(chunk, n_local)) if n_local else 1
        info["chunk_rows"] = chunk
        ptr = None
        for n, ptr in _slabs(produce, 0, n_local, chunk):
            _count(accs, n, ptr, n_cols, True, False)
        _merge_ranks(accs, world, rank, sums=True)
        states = [a.state() for a in accs]
        t0 = time.perf_counter()
        lo = [st["minmax"][0].astype(np.int64) for st in states]
        hi = [st["minmax"][1].astype(np.int64) for st in states]
        _set_windows(accs, lo, hi, budget_bytes, "shard")
        if n_local and n_local <= chunk:
            _count(accs, n_local, ptr, n_cols, False, True)
        elif n_local:
            info["reruns"] += 1
            for n, p in _slabs(produce, 0, n_local, chunk):
                _count(accs, n, p, n_cols, False, True)
        _merge_ranks(accs, world, rank, sums=False)
        out = []
        for a, st in zip(accs, states):
            if a.state(bins=False)["outside"].any():
                raise RuntimeError("shard: a value fell outside the [min, max] window of its column")
            col_ptr, value, count = a.export()
            out.append(dict(rows=st["rows"], moments=st["moments"], minmax=st["minmax"], col_ptr=col_ptr, value=value,
                            count=count))
        info["pass2_seconds"] += time.perf_counter() - t0
        return out
    finally:
        for a in accs:
            a.close()


def sparse_histogram(bins, lo, width):
    """(the numpy statement of ColumnAccumulator.export) dense unit-width bins of the windows [lo[a], lo[a] + width[a]) of every column, one after the other ->
    (col_ptr int64 [A+1], value uint32, count uint64): the non-zero bins of column a are entries col_ptr[a] ..
    col_ptr[a+1] - 1, in increasing value"""
    width = np.asarray(width, dtype=np.int64)
    off = np.concatenate([[0], np.cumsum(width)])
    bins = np.asarray(bins)[:int(off[-1])]
    nz = np.flatnonzero(bins)
    col = np.searchsorted(off, nz, side="right") - 1
    col_ptr = np.searchsorted(col, np.arange(len(width) + 1), side="left").astype(np.int64)
    value = (np.asarray(lo, dtype=np.int64)[col] + (nz - off[col])).astype(np.uint32)
    return col_ptr, value, bins[nz].astype(np.uint64)


def rebase_histogram(col_ptr, value, count, lo, width):
    """(the numpy statement of ColumnAccumulator.add_sparse into cleared bins) a sparse histogram (sparse_histogram)
    -> the dense uint32 bins of the windows [lo[a], lo[a] + width[a]), which must hold its values"""
    lo = np.asarray(lo, dtype=np.int64)
    width = np.asarray(width, dtype=np.int64)
    off = np.concatenate([[0], np.cumsum(width)])
    col = np.repeat(np.arange(len(width)), np.diff(np.asarray(col_ptr, dtype=np.int64)))
    pos = np.asarray(value, dtype=np.int64) - lo[col]
    if len(pos) and ((pos < 0) | (pos >= width[col])).any():
        raise ValueError("histogram values outside the windows they are rebased into")
    bins = np.zeros(max(int(off[-1]), 1), dtype=np.uint32)
    bins[off[col] + pos] = np.asarray(count, dtype=np.uint64)
    return bins


def _union(ctx, n_samples, observed, ref_fold, states, budget_bytes):
    """one accumulator holding the union of shard_states: the windows [min, max] of the union, every shard's
    integers added (gatb_colacc_merge: the 128-bit sum of squares with its carry) and its sparse histogram added on
    the device (ColumnAccumulator.add_sparse).  The caller closes it."""
    A = len(observed)
    if budget_bytes is None:
        import torch
        budget_bytes = int(ARENA_FRACTION * torch.cuda.mem_get_info(ctx.device)[0])
    acc = device.ColumnAccumulator(ctx, A, n_samples, observed, ref_fold)
    try:
        lo = np.min([st["minmax"][0] for st in states], axis=0).astype(np.int64)
        hi = np.max([st["minmax"][1] for st in states], axis=0).astype(np.int64)
        _set_windows([acc], [lo], [hi], budget_bytes, "merge")
        for st in states:
            acc.merge(dict(rows=int(st["rows"]), moments=np.ascontiguousarray(st["moments"], dtype=np.uint64),
                           minmax=np.ascontiguousarray(st["minmax"], dtype=np.uint32)))
            acc.add_sparse(st["col_ptr"], st["value"], st["count"])
        return acc
    except BaseException:
        acc.close()
        raise


def merge_shard_states(ctx, n_samples, observed, ref_fold, states, pseudo_count=1.0, budget_bytes=None):
    """the statistics of one counter plane from the shard_states of shards whose rows together are all n_samples
    samples -> statistics dict as Context.column_stats returns it"""
    acc = _union(ctx, n_samples, observed, ref_fold, states, budget_bytes)
    try:
        stats, missed = acc.finish(pseudo_count)
        if missed.any():
            raise RuntimeError("shard merge: a CI rank missed the [min, max] window of its column")
        return stats
    finally:
        acc.close()


def combine_shard_states(ctx, n_samples, observed, ref_fold, states, budget_bytes=None):
    """the shard_states of shards whose rows are consecutive ranges of one run -> the shard_states of their union
    range: summed integers, union [min, max], and the histogram over the union's [min, max] exported from the device
    (the state a shard job over the union range would have counted)"""
    acc = _union(ctx, n_samples, observed, ref_fold, states, budget_bytes)
    try:
        st = acc.state(bins=False)
        col_ptr, value, count = acc.export()
        return dict(rows=st["rows"], moments=st["moments"], minmax=st["minmax"], col_ptr=col_ptr, value=value,
                    count=count)
    finally:
        acc.close()
