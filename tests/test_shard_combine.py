"""Combining shards and reading the run of the first k samples, without a GPU: the range rules of combineShards and
mergeShardPrefix on synthetic shard files, and their bodies (sparse export and sparse add included) on the
SIMT-emulated build of the kernels (tests/emu)."""
import os
import sys

import numpy as np
import pytest

from tests.test_shards import HostSlab, STATS, _file, matrices, write_fake

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))


@pytest.fixture(scope="module")
def emu_ctx():
    import emu_context
    c = emu_context.context()
    yield c
    c.close()


@pytest.fixture
def on_emu(emu_ctx, monkeypatch):
    """the shard functions' context is the emulated one, and the arena budget does not ask a device"""
    import torch
    from gat_b200 import engine
    monkeypatch.setattr(engine, "getContext", lambda device=None: emu_ctx)
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (1 << 32, 1 << 32))
    return emu_ctx


# ------------------------------------------------------------------------------------------------ range rules
@pytest.mark.parametrize("case,ranges,named", [
    ("gap", [(0, 5), (6, 20)], 1), ("overlap", [(0, 6), (5, 20)], 1), ("duplicate", [(3, 10), (3, 10)], 1),
    ("empty", [(0, 5), (5, 5)], 1), ("past_end", [(10, 21)], 0)])
def test_combine_refuses(tmp_path, case, ranges, named):
    from gat_b200 import shards
    files = [write_fake(tmp_path / ("s%i.npz" % i), b, e) for i, (b, e) in enumerate(ranges)]
    out = str(tmp_path / "out.npz")
    with pytest.raises(ValueError) as e:
        shards.combineShards(files, out)
    assert os.path.basename(files[named]) in str(e.value), str(e.value)
    assert not os.path.exists(out)


def test_combine_and_prefix_refuse_shards_of_other_runs(tmp_path):
    from gat_b200 import shards
    files = [write_fake(tmp_path / "a.npz", 0, 5), write_fake(tmp_path / "b.npz", 5, 20, seed=np.uint64(12))]
    for call in (lambda: shards.combineShards(files, str(tmp_path / "out.npz")),
                 lambda: shards.mergeShardPrefix(files)):
        with pytest.raises(ValueError, match="seed") as e:
            call()
        assert "b.npz" in str(e.value)
    with pytest.raises(ValueError, match="no shard files"):
        shards.combineShards([], str(tmp_path / "out.npz"))
    with pytest.raises(ValueError, match="no shard files"):
        shards.mergeShardPrefix([])


@pytest.mark.parametrize("ranges,message,named", [
    ([(1, 5), (5, 20)], r"samples \[0, 1\) are in no shard", 0),
    ([(0, 6), (5, 9), (12, 20)], "overlap", 1),
    ([(0, 5), (12, 20), (10, 13)], "overlap", 1)])
def test_prefix_refuses(tmp_path, ranges, message, named):
    from gat_b200 import shards
    files = [write_fake(tmp_path / ("s%i.npz" % i), b, e) for i, (b, e) in enumerate(ranges)]
    with pytest.raises(ValueError, match=message) as e:
        shards.mergeShardPrefix(files)
    assert os.path.basename(files[named]) in str(e.value), str(e.value)


def test_combine_of_synthetic_shards(tmp_path, on_emu):
    """a contiguous range that does not start at 0, given in any order: metadata and rows kept, integers summed,
    min / max of the union, the histograms added"""
    from gat_b200 import shards
    files = [write_fake(tmp_path / ("s%i.npz" % i), b, e) for i, (b, e) in enumerate([(7, 12), (3, 7)])]
    out = str(tmp_path / "out.npz")
    shards.combineShards(files, out)
    got, first = shards.Shard(out), shards.Shard(files[0])
    assert (got.begin, got.end) == (3, 12)
    for k, v in first.arrays.items():
        if k != "sample_range" and not k.startswith("state_"):
            assert shards._same(got.arrays[k], v), k
    for ci in range(2):
        st, parts = got.state(0, ci), [shards.Shard(f).state(0, ci) for f in files]
        assert int(st["rows"]) == 10
        assert np.array_equal(st["moments"], parts[0]["moments"] + parts[1]["moments"])
        assert np.array_equal(st["minmax"], parts[0]["minmax"])
        assert np.array_equal(st["col_ptr"], np.arange(4)) and np.array_equal(st["value"], np.zeros(3))
        assert np.array_equal(st["count"], np.full(3, 10)) and st["count"].dtype == np.uint64
    # a combined file is an ordinary shard
    assert [s.end for s in shards.readShards([write_fake(tmp_path / "head.npz", 0, 3), out,
                                              write_fake(tmp_path / "tail.npz", 12, 20)])] == [3, 12, 20]


# ------------------------------------------------------------------------------------------ emulated kernels
def _shard_files(ctx, tmp_path, tag, mats, obs, ref, ranges, chunk=8):
    from gat_b200 import matrixfree
    S, A = mats.shape[1], mats.shape[2]
    files = []
    for k, (b, e) in enumerate(ranges):
        states = matrixfree.shard_states(ctx, HostSlab(mats[:, b:e], chunk), [(obs[i], ref) for i in range(2)], S,
                                         e - b, A, chunk, budget_bytes=1 << 30)
        files.append(_file(tmp_path / ("%s%i.npz" % (tag, k)), S, (b, e), obs, ref, states))
    return files


def _stats(results, i):
    name = ["nucleotide-overlap", "segment-overlap"][i]
    return dict((k, np.array([getattr(r, k) for r in results if r.counter == name])) for k in STATS)


@pytest.mark.parametrize("S,A,whole,pieces,with_ref", [
    (41, 9, (5, 41), [(30, 41), (5, 13), (13, 30)], False),
    (97, 30, (0, 60), [(40, 60), (0, 1), (20, 40), (1, 20)], True)])
def test_combined_shards_on_the_emulated_kernels(on_emu, tmp_path, S, A, whole, pieces, with_ref):
    """combineShards of pieces of [b, e) == the shard file of one job over [b, e), array by array; a tree of
    combined files merges to gatb_column_stats of the whole matrix"""
    from gat_b200 import shards
    rng = np.random.default_rng(S)
    mats, obs = matrices(rng, S, A)
    ref = rng.choice([0.01, 0.5, 1.0, 3.0, 1000.0], A) if with_ref else None
    single = _shard_files(on_emu, tmp_path, "single", mats, obs, ref, [whole])[0]
    parts = _shard_files(on_emu, tmp_path, "part", mats, obs, ref, pieces)
    out = str(tmp_path / "combined.npz")
    shards.combineShards(parts, out)
    want, got = shards.Shard(single).arrays, shards.Shard(out).arrays
    assert sorted(want) == sorted(got)
    for k in want:
        assert want[k].dtype == got[k].dtype and shards._same(want[k], got[k]), k
    # the tree: the two lowest pieces first, then that file with the rest, then the whole run
    by_range = [p for _, p in sorted(zip(pieces, parts))]
    left, tree = str(tmp_path / "left.npz"), str(tmp_path / "tree.npz")
    shards.combineShards(by_range[:2], left)
    shards.combineShards(by_range[2:] + [left], tree)
    assert all(shards._same(shards.Shard(tree).arrays[k], want[k]) for k in want)
    outside = [r for r in [(0, whole[0]), (whole[1], S)] if r[0] < r[1]]
    others = _shard_files(on_emu, tmp_path, "other", mats, obs, ref, outside)
    merged = shards._merge(shards.readShards([tree] + others), on_emu, budget_bytes=1 << 30)
    for i in range(2):
        st = on_emu.column_stats(mats[i], obs[i], pseudo_count=1.0, ref_fold=ref)
        for k in STATS:
            assert np.array_equal(_stats(merged, i)[k], st[k]), (i, k)


@pytest.mark.parametrize("ranges,k", [([(0, 13), (13, 20), (25, 41)], 20), ([(30, 41), (0, 3)], 3),
                                      ([(20, 41), (0, 7), (7, 20)], 41)])
def test_prefix_on_the_emulated_kernels(on_emu, tmp_path, capsys, ranges, k):
    """the shards that tile [0, k) read as the statistics of the first k samples (the CI ranks of k); the shards
    past the gap are named on stderr"""
    from gat_b200 import shards
    S, A = 41, 9
    rng = np.random.default_rng(5)
    mats, obs = matrices(rng, S, A)
    files = _shard_files(on_emu, tmp_path, "p", mats, obs, None, ranges)
    got_k, results = shards.mergeShardPrefix(files)
    assert got_k == k and results[0].nsamples == k
    for i in range(2):
        st = on_emu.column_stats(mats[i, :k], obs[i], pseudo_count=1.0)
        for key in STATS:
            assert np.array_equal(_stats(results, i)[key], st[key]), (i, key)
    err = capsys.readouterr().err
    for f, (b, e) in zip(files, ranges):
        assert (os.path.basename(f) in err) == (b >= k)


def test_add_sparse_and_export_on_the_emulated_kernels(emu_ctx):
    """the device sparse add against rebase_histogram, its refusal leaving the bins alone, and the device export
    against sparse_histogram, on wide windows and counts near 2^32"""
    from gat_b200 import device, matrixfree
    rng = np.random.default_rng(3)
    A = 7
    lo = rng.integers(0, 1000, A)
    width = np.array([1, 600, 3, 1, 257, 40, 2])
    dense = np.concatenate([rng.integers(0, 3, w) * (rng.random(w) < 0.4) for w in width]).astype(np.uint32)
    dense[width[0]:width[0] + 4] = 0xffffffff - np.arange(4, dtype=np.uint32)     # column 1: total past 2^32
    col_ptr, value, count = matrixfree.sparse_histogram(dense, lo, width)
    acc = device.ColumnAccumulator(emu_ctx, A, 100, np.zeros(A))
    try:
        lo2, width2 = np.maximum(lo - 5, 0), width + 9
        acc.set_windows(lo2, width2)
        acc.add_sparse(col_ptr, value, count)
        want = matrixfree.rebase_histogram(col_ptr, value, count, lo2, width2)
        assert np.array_equal(acc.state()["bins"], want)
        with pytest.raises(ValueError, match="outside"):
            acc.add_sparse(col_ptr, value + np.uint32(50), count)
        with pytest.raises(ValueError, match="outside"):
            acc.add_sparse(col_ptr, value, count + np.uint64(1 << 32))
        assert np.array_equal(acc.state()["bins"], want)
        got = acc.export()
        exp = matrixfree.sparse_histogram(want, lo2, width2)
        for g, w in zip(got, exp):
            assert g.dtype == w.dtype and np.array_equal(g, w)
        assert np.array_equal(got[2], count) and np.array_equal(got[1], value)
    finally:
        acc.close()
