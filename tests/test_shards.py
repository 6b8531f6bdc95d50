"""Sharded runs without a GPU: the shard rules of the run plan, the checks of mergeShards on synthetic shard files,
the sparse histograms, and the shard accumulation and merge on the SIMT-emulated build of the kernels (tests/emu)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))

STATS = ["expected", "stddev", "lower95", "upper95", "fold", "pvalue"]


@pytest.fixture
def plan(monkeypatch):
    """_planRun of a shard job; a device query or a collective inside it fails the test"""
    import torch
    import torch.distributed
    from gat_b200 import _planRun

    def refuse(*args, **kw):
        raise AssertionError("the run plan queried a device or ran a collective")
    for name in ("mem_get_info", "synchronize", "current_stream", "set_device", "device_count"):
        monkeypatch.setattr(torch.cuda, name, refuse)
    for name in ("all_gather_object", "broadcast_object_list", "all_gather", "barrier"):
        monkeypatch.setattr(torch.distributed, name, refuse)

    def make(**kw):
        args = dict(num_samples=1000, n_tracks=1, n_annotations=10, counter_names=["nucleotide-overlap"],
                    counts_table=False, keep_samples=None, exchange="auto", transport="peer", rank=0, world=1,
                    free_bytes=0, sample_range=(0, 1000), seeded=True)
        args.update(kw)
        return _planRun(**args)
    return make


# ---------------------------------------------------------------------------------------------- the plan
@pytest.mark.parametrize("world", [1, 2, 8])
@pytest.mark.parametrize("S,begin,end", [(1000, 0, 1000), (1000, 1, 4096 // 8), (4097, 4096, 4097), (20, 3, 10)])
def test_shard_rows_tile_the_range(plan, world, S, begin, end):
    rows = []
    for rank in range(world):
        p = plan(num_samples=S, sample_range=(begin, end), rank=rank, world=world, keep_samples=None)
        assert p.matrix_free and p.columns == (0, 10)
        rows.append(p.rows)
    assert rows[0][0] == begin and rows[-1][1] == end
    assert all(rows[r][1] == rows[r + 1][0] for r in range(world - 1))
    assert all(b <= e for b, e in rows)
    # a shard is always counted by the accumulators, whatever the default mode or the matrix sizes would say
    assert plan(num_samples=S, sample_range=(begin, end), keep_samples=False, free_bytes=1 << 50).matrix_free


@pytest.mark.parametrize("world", [1, 2, 8])
def test_shard_refusals(plan, world):
    with pytest.raises(ValueError, match="output_counts_pattern"):
        plan(counts_table=True, world=world)
    with pytest.raises(ValueError, match="keep_samples=True"):
        plan(keep_samples=True, world=world)
    for bad in ((0, 0), (5, 3), (-1, 10), (0, 1001), (1000, 1001)):
        with pytest.raises(ValueError, match="sample_range"):
            plan(sample_range=bad, world=world)
    with pytest.raises(ValueError, match="sample_range"):
        plan(num_samples=1 << 32, sample_range=(0, 10), world=world)
    with pytest.raises(NotImplementedError, match="nucleotide-density"):
        plan(counter_names=["nucleotide-overlap", "nucleotide-density"], world=world)
    with pytest.raises(ValueError, match="seeded"):
        plan(seeded=False, world=world)
    # the range is the shard's business: run()'s plan is unchanged without one
    assert not plan(sample_range=None, keep_samples=True, world=world).matrix_free


# ------------------------------------------------------------------------------------------ sparse histograms
def test_sparse_histogram_and_rebase_against_numpy():
    from gat_b200 import matrixfree
    rng = np.random.default_rng(7)
    A = 23
    lo = rng.integers(0, 1000, A)
    width = rng.integers(1, 60, A)
    width[3] = 1
    bins = np.concatenate([rng.integers(0, 4, w) * (rng.random(w) < 0.5) for w in width]).astype(np.uint32)
    bins[0] = 0
    col_ptr, value, count = matrixfree.sparse_histogram(bins, lo, width)
    # restatement: column by column, the non-zero bins in increasing value
    off = np.concatenate([[0], np.cumsum(width)])
    want_v, want_c, want_p = [], [], [0]
    for a in range(A):
        b = bins[off[a]:off[a + 1]]
        for i in range(len(b)):
            if b[i]:
                want_v.append(lo[a] + i)
                want_c.append(b[i])
        want_p.append(len(want_v))
    assert col_ptr.dtype == np.int64 and value.dtype == np.uint32 and count.dtype == np.uint64
    assert np.array_equal(col_ptr, want_p) and np.array_equal(value, want_v) and np.array_equal(count, want_c)
    # rebased into wider windows (the union of several shards'): the same counts at the same values
    lo2 = np.maximum(lo - rng.integers(0, 20, A), 0)
    width2 = width + (lo - lo2) + rng.integers(0, 20, A)
    dense = matrixfree.rebase_histogram(col_ptr, value, count, lo2, width2)
    off2 = np.concatenate([[0], np.cumsum(width2)])
    want = np.zeros(int(off2[-1]), dtype=np.uint32)
    for a in range(A):
        for i in range(width[a]):
            want[off2[a] + lo[a] - lo2[a] + i] = bins[off[a] + i]
    assert np.array_equal(dense, want)
    # rebased into its own windows: the dense bins themselves
    assert np.array_equal(matrixfree.rebase_histogram(col_ptr, value, count, lo, width), bins)
    with pytest.raises(ValueError):
        matrixfree.rebase_histogram(col_ptr, value, count, lo + 1, width)


# ----------------------------------------------------------------------------------------- shard files
def fake_state(rng, A):
    col_ptr = np.arange(A + 1, dtype=np.int64)
    return dict(rows=np.int64(5), moments=rng.integers(0, 99, (5, A)).astype(np.uint64),
                minmax=np.stack([np.zeros(A), np.full(A, 9)]).astype(np.uint32), col_ptr=col_ptr,
                value=np.zeros(A, dtype=np.uint32), count=np.full(A, 5, dtype=np.uint64))


def write_fake(path, begin, end, S=20, **change):
    """a synthetic shard file of one track, two counters and three annotations"""
    from gat_b200 import shards
    rng = np.random.default_rng(0)
    A, C = 3, 2
    out = dict(format=np.array(shards.FORMAT), version=np.int64(shards.FORMAT_VERSION), seed=np.uint64(11),
               num_samples=np.int64(S), sample_range=np.array([begin, end], dtype=np.int64),
               pseudo_count=np.float64(1.0), has_reference=np.bool_(False),
               counters=np.array(["nucleotide-overlap", "segment-overlap"]), tracks=np.array(["merged"]),
               annotations=np.array(["a", "b", "c"]), digest=np.array("0" * 64))
    out["row_counter"] = np.repeat(np.arange(C), A).astype(np.int64)
    out["row_track"] = np.zeros(A * C, dtype=np.int64)
    out["row_annotation"] = np.tile(np.arange(A), C).astype(np.int64)
    out["row_observed"] = np.arange(A * C, dtype=np.float64)
    out["row_ref_fold"] = np.full(A * C, np.nan)
    for k in shards.SIZES:
        out["row_" + k] = np.arange(A * C, dtype=np.int64) + 100
    for ci in range(C):
        for k, v in fake_state(rng, A).items():
            out["state_0_%i_%s" % (ci, k)] = v
    out.update(change)
    shards._save(str(path), out)
    return str(path)


def test_merge_accepts_any_order_of_a_tiling(tmp_path):
    from gat_b200 import shards
    files = [write_fake(tmp_path / ("s%i.npz" % i), b, e) for i, (b, e) in enumerate([(7, 20), (0, 1), (1, 7)])]
    got = shards.readShards(files)
    assert sorted((s.begin, s.end) for s in got) == [(0, 1), (1, 7), (7, 20)]
    assert got[0].counters == ["nucleotide-overlap", "segment-overlap"] and got[0].tracks == ["merged"]
    assert shards.readShards([write_fake(tmp_path / "all.npz", 0, 20)])[0].num_samples == 20


@pytest.mark.parametrize("case", ["gap_inside", "gap_start", "gap_end", "overlap", "duplicate", "seed", "digest",
                                  "counters", "tracks", "annotations", "num_samples", "pseudo_count", "reference",
                                  "observed", "sizes", "version", "not_npz", "npz_not_shard", "none"])
def test_merge_refuses(tmp_path, case):
    from gat_b200 import shards
    ranges = {"gap_inside": [(0, 5), (6, 20)], "gap_start": [(1, 20)], "gap_end": [(0, 5), (5, 19)],
              "overlap": [(0, 6), (5, 20)], "duplicate": [(0, 10), (0, 10), (10, 20)]}.get(case, [(0, 10), (10, 20)])
    change = dict(seed=dict(seed=np.uint64(12)), digest=dict(digest=np.array("1" * 64)),
                  counters=dict(counters=np.array(["nucleotide-overlap", "segment-midoverlap"])),
                  tracks=dict(tracks=np.array(["other"])), annotations=dict(annotations=np.array(["a", "b", "d"])),
                  num_samples=dict(num_samples=np.int64(21)), pseudo_count=dict(pseudo_count=np.float64(0.5)),
                  reference=dict(has_reference=np.bool_(True)),
                  observed=dict(row_observed=np.arange(6, dtype=np.float64) + 1),
                  sizes=dict(row_overlap_size=np.arange(6, dtype=np.int64)),
                  version=dict(version=np.int64(shards.FORMAT_VERSION + 1))).get(case, {})
    files = [write_fake(tmp_path / ("s%i.npz" % i), b, e, **(change if i == len(ranges) - 1 else {}))
             for i, (b, e) in enumerate(ranges)]
    if case == "not_npz":
        files[-1] = str(tmp_path / "table.tsv")
        with open(files[-1], "w") as f:
            f.write("track\tannotation\n")
    if case == "npz_not_shard":
        files[-1] = str(tmp_path / "other.npz")
        np.savez(files[-1], x=np.zeros(3))
    if case == "none":
        files = []
    with pytest.raises(ValueError) as e:
        shards.readShards(files)
    if case not in ("gap_start", "none"):
        named = files[1] if case == "duplicate" else files[-1]          # (the second of the two [0, 10) shards)
        assert os.path.basename(named) in str(e.value), str(e.value)


# ---------------------------------------------------------------------------------- emulated kernels
@pytest.fixture(scope="module")
def emu_ctx():
    import emu_context
    c = emu_context.context()
    yield c
    c.close()


class HostSlab(object):
    """the slab of the emulated build ("device" memory is host memory there); counts its calls"""

    def __init__(self, mats, chunk):
        self.mats = mats
        self.buf = np.zeros(mats.shape[0] * chunk * mats.shape[2], dtype=np.uint32)
        self.calls = 0

    def __call__(self, r0, n):
        P, _, A = self.mats.shape
        self.calls += 1
        self.buf[:P * n * A] = self.mats[:, r0:r0 + n].reshape(-1)
        return self.buf.ctypes.data


def matrices(rng, S, A):
    """two planes; column 0 of plane 0 near 2^32, so that the shards' sums of squares carry past 2^64"""
    mats = (rng.integers(0, 1000, A)[None, None, :] + rng.integers(0, 300, (2, S, A))).astype(np.uint32)
    mats[0, :, 0] = 0xffffffff - rng.integers(0, 3, S).astype(np.uint32)
    obs = np.stack([np.asarray(mats[i, S // 2], dtype=np.float64) + [0.5, 0.0][i] for i in range(2)])
    obs[0, 0] = 4294967294.0
    return mats, obs


@pytest.mark.parametrize("S,A,ranges,chunk,with_ref", [
    (1, 5, [(0, 1)], 1, False),
    (20, 9, [(0, 1), (1, 19), (19, 20)], 4, True),
    (41, 9, [(30, 41), (0, 13), (13, 30)], 64, False),
    (97, 30, [(0, 20), (20, 40), (40, 60), (60, 80), (80, 97)], 7, True)])
def test_shards_merge_to_the_statistics_of_the_matrix_on_the_emulated_kernels(emu_ctx, tmp_path, S, A, ranges, chunk,
                                                                              with_ref):
    """shard_states of each range (a slab smaller than the range samples pass 2 again, one that holds it does not),
    merged through shard files == gatb_column_stats of the whole matrix, with == and 128-bit carries"""
    from gat_b200 import matrixfree, shards
    rng = np.random.default_rng(S)
    mats, obs = matrices(rng, S, A)
    ref = rng.choice([0.01, 0.5, 1.0, 3.0, 1000.0], A) if with_ref else None
    want = [emu_ctx.column_stats(mats[i], obs[i], pseudo_count=1.0, ref_fold=ref) for i in range(2)]
    files = []
    for k, (b, e) in enumerate(ranges):
        slab = HostSlab(mats[:, b:e], chunk)
        reruns = matrixfree.info["reruns"]
        states = matrixfree.shard_states(emu_ctx, slab, [(obs[i], ref) for i in range(2)], S, e - b, A, chunk,
                                         budget_bytes=1 << 30)
        fits = e - b <= chunk
        assert slab.calls == (1 if fits else 2 * -(-(e - b) // chunk))
        assert matrixfree.info["reruns"] - reruns == (0 if fits else 1)
        st0 = states[0]
        assert st0["rows"] == e - b and st0["moments"][3:].dtype == np.uint64
        assert np.array_equal(st0["minmax"], np.stack([mats[0, b:e].min(axis=0), mats[0, b:e].max(axis=0)]))
        for i, st in enumerate(states):
            col = np.repeat(np.arange(A), np.diff(st["col_ptr"]))
            for a in range(A):
                v, c = np.unique(mats[i, b:e, a], return_counts=True)
                assert np.array_equal(st["value"][col == a], v) and np.array_equal(st["count"][col == a], c)
        files.append(_file(tmp_path / ("s%i.npz" % k), S, (b, e), obs, ref, states))
    sq = [shards.Shard(f).state(0, 0)["moments"] for f in files]
    assert S == 1 or sum((int(m[4][0]) << 64) + int(m[3][0]) for m in sq) >= 1 << 64   # (column 0: past 2^64)
    got = shards._merge(shards.readShards(files[::-1]), emu_ctx, budget_bytes=1 << 30)
    for i in range(2):
        for k in STATS:
            g = np.array([getattr(r, k) for r in got if r.counter == ["nucleotide-overlap", "segment-overlap"][i]])
            assert np.array_equal(g, want[i][k]), (i, k, g, want[i][k])
    assert len(got) == 2 * A and got[0].nsamples == S
    with pytest.raises(RuntimeError, match="keep_samples=True"):
        got[0].samples


def _file(path, S, rng_, obs, ref, states):
    """a shard file of one track "t", two counters and the annotation columns of obs"""
    from gat_b200 import shards
    A = obs.shape[1]
    out = dict(format=np.array(shards.FORMAT), version=np.int64(shards.FORMAT_VERSION), seed=np.uint64(1),
               num_samples=np.int64(S), sample_range=np.array(rng_, dtype=np.int64), pseudo_count=np.float64(1.0),
               has_reference=np.bool_(ref is not None), counters=np.array(["nucleotide-overlap", "segment-overlap"]),
               tracks=np.array(["t"]), annotations=np.array(["a%i" % a for a in range(A)]),
               digest=np.array("0" * 64))
    out["row_counter"] = np.repeat(np.arange(2), A).astype(np.int64)
    out["row_track"] = np.zeros(2 * A, dtype=np.int64)
    out["row_annotation"] = np.tile(np.arange(A), 2).astype(np.int64)
    out["row_observed"] = obs.reshape(-1).astype(np.float64)
    out["row_ref_fold"] = np.tile(ref, 2) if ref is not None else np.full(2 * A, np.nan)
    for k in shards.SIZES:
        out["row_" + k] = np.full(2 * A, 10, dtype=np.int64)
    for ci, st in enumerate(states):
        for k in shards.STATE:
            out["state_0_%i_%s" % (ci, k)] = np.asarray(st[k])
    shards._save(str(path), out)
    return str(path)
