"""Combining shards and reading the run of the first k samples on the GPU: the device export and sparse add of the
column accumulator against their numpy statements, combineShards against one shard job over the same range, trees
of combined files and mergeShardPrefix against run(), compared with ==."""
import os
import random

import numpy as np
import pytest

from tests.test_gpu_shards import (BATCH, INTEGER_COUNTERS, SAMPLERS, Fold, assert_runs_identical, cli_tables,
                                   output_args, problem, run_shards, run_whole, write_inputs)

SLAB_ROWS = 1500


@pytest.fixture
def small_slabs(monkeypatch):
    """slabs of 1500 rows: larger shards sample their histogram pass again, smaller ones read it from the slab"""
    from gat_b200 import matrixfree
    monkeypatch.setattr(matrixfree, "SLAB_BYTES", 4 * len(INTEGER_COUNTERS) * 7 * SLAB_ROWS)


def filled(ctx, lo, width, columns):
    """an accumulator with the windows (lo, width) whose histograms hold the rows of `columns` [rows][A] (uint32),
    counted on the device"""
    import torch
    from gat_b200 import device
    A = len(lo)
    acc = device.ColumnAccumulator(ctx, A, max(1, columns.shape[0]), np.zeros(A))
    acc.set_windows(lo, width)
    if columns.shape[0]:
        dev = torch.from_numpy(np.ascontiguousarray(columns).view(np.int32)).cuda()
        acc.add(dev.data_ptr(), columns.shape[0], sums=False, hist=True)
        torch.cuda.synchronize()
    return acc


def check_export(acc, lo, width):
    from gat_b200 import matrixfree
    want = matrixfree.sparse_histogram(acc.state()["bins"], lo, width)
    got = acc.export()
    for g, w in zip(got, want):
        assert g.dtype == w.dtype and np.array_equal(g, w)
    return got


@pytest.mark.gpu
def test_export_against_sparse_histogram(ctx):
    """columns with one value, all-zero columns, windows much wider than a CTA's tile of 256 bins, sparse and dense"""
    rng = np.random.default_rng(1)
    A, S = 300, 3000
    lo = rng.integers(0, 1 << 20, A).astype(np.int64)
    width = rng.integers(1, 3000, A)
    width[:5] = [1, 256, 257, 100000, 511]
    cols = (lo[None, :] + (rng.random((S, A)) ** 3 * width[None, :])).astype(np.uint32)
    cols[:, 10] = lo[10] + 7 if width[10] > 7 else lo[10]                   # one value
    cols[:, 11] = lo[11] + width[11] + 5                                    # above the window: all bins zero
    cols[:, 12] = max(lo[12] - 1, 0) if lo[12] else lo[12] + width[12]      # below (or above): all zero
    acc = filled(ctx, lo, width, cols)
    try:
        col_ptr, value, count = check_export(acc, lo, width)
        assert col_ptr[11] == col_ptr[12] == col_ptr[13] and col_ptr[11] - col_ptr[10] == 1 and count[col_ptr[10]] == S
        assert int(count.sum()) + int(acc.state(bins=False)["outside"].sum()) == S * A
    finally:
        acc.close()
    # no values at all, and one column of one bin
    for A_, w_ in ((5, 40), (1, 1)):
        acc = filled(ctx, np.zeros(A_, dtype=np.int64), np.full(A_, w_), np.zeros((0, A_), dtype=np.uint32))
        try:
            col_ptr, value, count = check_export(acc, np.zeros(A_, dtype=np.int64), np.full(A_, w_))
            assert not col_ptr.any() and len(value) == 0 and len(count) == 0
        finally:
            acc.close()


@pytest.mark.gpu
def test_add_sparse_against_rebase_and_counts_near_two_to_the_32(ctx):
    """add_sparse == rebase_histogram into wider windows; bins near 2^32 (column totals past 2^32) export exactly;
    a value outside its window or a count of 2^32 is refused and leaves the bins as they were"""
    from gat_b200 import device, matrixfree
    rng = np.random.default_rng(2)
    A = 400
    lo = rng.integers(0, 100000, A).astype(np.int64)
    width = rng.integers(1, 2000, A)
    width[0] = 70000
    dense = np.concatenate([rng.integers(0, 5, w) * (rng.random(w) < 0.3) for w in width]).astype(np.uint32)
    dense[:300] = 0xffffffff - np.arange(300, dtype=np.uint32)                # column 0: total far past 2^32
    col_ptr, value, count = matrixfree.sparse_histogram(dense, lo, width)
    acc = device.ColumnAccumulator(ctx, A, 100, np.zeros(A))
    try:
        lo2 = np.maximum(lo - rng.integers(0, 50, A), 0)
        width2 = width + (lo - lo2) + rng.integers(0, 50, A)
        acc.set_windows(lo2, width2)
        acc.add_sparse(col_ptr, value, count)
        want = matrixfree.rebase_histogram(col_ptr, value, count, lo2, width2)
        assert np.array_equal(acc.state()["bins"], want)
        got = check_export(acc, lo2, width2)
        assert np.array_equal(got[1], value) and np.array_equal(got[2], count)
        for bad in ((value + np.uint32(100000), count), (np.where(np.arange(len(value)) == 7, lo2[0] - 1 if lo2[0]
                                                                  else 0xffffffff, value).astype(np.uint32), count),
                    (value, np.where(np.arange(len(count)) == 3, np.uint64(1 << 32), count))):
            with pytest.raises(ValueError, match="outside"):
                acc.add_sparse(col_ptr, *bad)
            assert np.array_equal(acc.state()["bins"], want)
        # the same histogram twice: doubled (the bins are uint32, and no bin here passes 2^32 - 1 twice over)
        half = count.copy()
        half[:300] = 1
        acc.set_windows(lo2, width2)
        acc.add_sparse(col_ptr, value, half)
        acc.add_sparse(col_ptr, value, half)
        assert np.array_equal(acc.state()["bins"], matrixfree.rebase_histogram(col_ptr, value, 2 * half, lo2, width2))
    finally:
        acc.close()


@pytest.mark.gpu
def test_shard_file_arrays_equal_the_numpy_export(tmp_path, monkeypatch, small_slabs):
    """every histogram a shard job exports from the device is the one sparse_histogram makes of the dense bins of
    the same accumulator: the arrays the host path wrote before, for a job that reads its slab and one that
    samples again"""
    from gat_b200 import device, matrixfree
    export = device.ColumnAccumulator.export
    checked = []

    def both(self):
        got = export(self)
        st = self.state()
        lo = st["minmax"][0].astype(np.int64)
        want = matrixfree.sparse_histogram(st["bins"], lo, st["minmax"][1].astype(np.int64) - lo + 1)
        for g, w in zip(got, want):
            assert g.dtype == w.dtype and np.array_equal(g, w)
        checked.append(int(got[0][-1]))
        return got
    monkeypatch.setattr(device.ColumnAccumulator, "export", both)
    inputs = problem(False)
    run_shards(tmp_path, "x", inputs, SAMPLERS["annotator"], 5000, [(0, 1000), (1000, 5000)])
    assert len(checked) == 2 * 2 * len(INTEGER_COUNTERS) and min(checked) > 0


CASES = [("annotator", False, False), ("annotator", True, True), ("segments", True, False), ("shift", False, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("sampler,isochores,with_ref", CASES)
def test_combined_shards_equal_one_job_and_merge_to_the_run(tmp_path, small_slabs, sampler, isochores, with_ref):
    """combineShards of 2, 3 and 5 shuffled uneven pieces of [b, e) == runShard over [b, e), array by array; the
    combined files, merged as a tree, == mergeShards of the original shards == run()"""
    import gat_b200
    from gat_b200 import shards
    inputs = problem(isochores)
    reference = None
    if with_ref:
        folds = [0.01, 0.5, 1.0, 2.0, 1000.0, 0.25, 4.0]
        reference = dict((t, dict((a, Fold(folds[i % len(folds)])) for i, a in enumerate(inputs[1].tracks)))
                         for t in inputs[0].tracks)
    S = 3 * BATCH + 5
    b, e = 1000, S - 2
    whole = run_whole(inputs, SAMPLERS[sampler], S, reference)
    single = run_shards(tmp_path, "single", inputs, SAMPLERS[sampler], S, [(b, e)], reference)[0]
    outside = run_shards(tmp_path, "out", inputs, SAMPLERS[sampler], S, [(0, b), (e, S)], reference)
    want = shards.Shard(single).arrays
    tops = []
    for k, cuts in ((2, [b, b + 1, e]), (3, [b, 5000, 5001, e]), (5, [b, b + 3, 2 * BATCH, 2 * BATCH + 1, e - 1, e])):
        pieces = run_shards(tmp_path, "k%i" % k, inputs, SAMPLERS[sampler], S, list(zip(cuts[:-1], cuts[1:])),
                            reference)
        out = str(tmp_path / ("combined%i.npz" % k))
        gat_b200.combineShards(pieces, out)
        got = shards.Shard(out).arrays
        assert sorted(got) == sorted(want)
        for key in want:
            assert got[key].dtype == want[key].dtype and shards._same(got[key], want[key]), (k, key)
        # a tree: pairs of neighbours first, then those files together with the whole run's other shards
        order = sorted(pieces, key=lambda f: shards.Shard(f).begin)
        level = []
        for i in range(0, len(order), 2):
            f = str(tmp_path / ("k%i_pair%i.npz" % (k, i)))
            gat_b200.combineShards(order[i:i + 2], f)
            level.append(f)
        top = str(tmp_path / ("k%i_top.npz" % k))
        gat_b200.combineShards(level[::-1] + outside, top)
        tops.append(top)
        assert_runs_identical(whole, gat_b200.mergeShards([top]))
        originals = outside + pieces
        random.Random(k).shuffle(originals)
        assert_runs_identical(whole, gat_b200.mergeShards(originals))
    assert_runs_identical(whole, gat_b200.mergeShards(outside + [str(tmp_path / "combined3.npz")]))


@pytest.mark.gpu
@pytest.mark.parametrize("sampler,isochores", [("annotator", False), ("segments", True), ("shift", True)])
def test_prefix_equals_the_run_of_the_first_k_samples(tmp_path, small_slabs, capsys, sampler, isochores):
    """shards missing after k: == run(num_samples=k), for k inside one slab and k across several; every shard there:
    == mergeShards; the refusals"""
    import gat_b200
    inputs = problem(isochores)
    S = 3 * BATCH + 5
    cuts = [0, 700, 1100, 1400, 5000, 6000, 9000, S]
    files = run_shards(tmp_path, "p", inputs, SAMPLERS[sampler], S, list(zip(cuts[:-1], cuts[1:])))
    by_begin = dict((int(np.load(f)["sample_range"][0]), f) for f in files)
    for k, missing in ((1100, 1100), (5000, 5000)):
        present = [f for b, f in by_begin.items() if b != missing]
        got_k, results = gat_b200.mergeShardPrefix(present)
        assert got_k == k
        assert_runs_identical(run_whole(inputs, SAMPLERS[sampler], k), results)
        assert os.path.basename(by_begin[cuts[-2]]) in capsys.readouterr().err
    got_k, results = gat_b200.mergeShardPrefix(files)
    assert got_k == S
    assert_runs_identical(gat_b200.mergeShards(files), results)
    with pytest.raises(ValueError, match=r"samples \[0, 700\) are in no shard"):
        gat_b200.mergeShardPrefix([f for b, f in by_begin.items() if b != 0])
    other = run_shards(tmp_path, "o", inputs, SAMPLERS[sampler], S, [(600, 1200)])[0]
    with pytest.raises(ValueError, match="overlap") as e:
        gat_b200.mergeShardPrefix(files + [other])
    assert os.path.basename(other) in str(e.value)
    with pytest.raises(ValueError, match="gap"):
        gat_b200.mergeShards([f for b, f in by_begin.items() if b != 1100])


@pytest.mark.gpu
def test_cli_prefix_and_combine_print_the_tables_of_runs(tmp_path, capfd):
    """--prefix prints the table of the run of the first k samples and logs the range; --combine writes a shard
    and prints nothing; the tables are byte-identical to the runs'"""
    from gat_b200 import cli, shards
    S, k = 300, 180
    counters = ["nucleotide-overlap", "segment-overlap"]
    common = write_inputs(tmp_path, True) + ["--counter=" + c for c in counters] + ["--random-seed=7", "-v", "0"]
    assert cli.main(["gat-run"] + common + ["--num-samples=%i" % S] + output_args(tmp_path, "whole")) == 0
    assert cli.main(["gat-run"] + common + ["--num-samples=%i" % k] + output_args(tmp_path, "first")) == 0
    files = []
    for i, (b, e) in enumerate([(100, 180), (0, 100), (250, 300), (180, 250)]):
        f = str(tmp_path / ("part%i.npz" % i))
        assert cli.main(["gat-run"] + common + ["--num-samples=%i" % S, "--sample-range=%i:%i" % (b, e),
                                                "--output-shard=" + f]) == 0
        files.append(f)
    capfd.readouterr()
    assert shards.main(["gat-merge", "--prefix"] + output_args(tmp_path, "prefix") + files[:3]) == 0
    assert "samples [0, %i) of %i" % (k, S) in capfd.readouterr().err
    assert cli_tables(tmp_path, "prefix", [], counters) == cli_tables(tmp_path, "first", [], counters)
    combined = str(tmp_path / "combined.npz")
    assert shards.main(["gat-merge", "--combine=" + combined, files[3], files[0]]) == 0
    assert capfd.readouterr().out == ""
    assert shards.main(["gat-merge"] + output_args(tmp_path, "merged") + [files[2], combined, files[1]]) == 0
    assert cli_tables(tmp_path, "merged", [], counters) == cli_tables(tmp_path, "whole", [], counters)
