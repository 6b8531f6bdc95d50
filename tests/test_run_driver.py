"""gat_b200.run()'s driver: the run plan (_planRun) on injected sizes without a GPU, and on the GPU a track without
any unit and an empty workspace in the matrix and the matrix-free mode."""
import os
import re

import numpy as np
import pytest

INTEGER_COUNTERS = ["nucleotide-overlap", "segment-overlap", "segment-midoverlap", "annotation-overlap",
                    "annotation-midoverlap"]
STATS = ["expected", "stddev", "lower95", "upper95", "fold", "pvalue"]


@pytest.fixture
def plan(monkeypatch):
    """_planRun with defaults for every argument; a device query or a collective inside it fails the test"""
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
                    counts_table=False, keep_samples=True, exchange="auto", transport="peer", rank=0, world=1,
                    free_bytes=0)
        args.update(kw)
        return _planRun(**args)
    return make


# ---------------------------------------------------------------------------------------------- without a GPU
@pytest.mark.parametrize("world", [1, 2, 8])
def test_auto_exchange_switches_to_columns_at_one_gib(plan, world):
    """4 * S * A * counters bytes: 2^30 exactly at S = 262144, A = 512, two counters"""
    two = ["nucleotide-overlap", "segment-overlap"]
    big = plan(num_samples=262144, n_annotations=512, counter_names=two, world=world)
    small = plan(num_samples=262143, n_annotations=512, counter_names=two, world=world)
    assert big.exchange == ("columns" if world > 1 else "allgather")
    assert small.exchange == "allgather"
    # a counts table needs every column on rank 0: auto keeps the all-gather
    assert plan(num_samples=262144, n_annotations=512, counter_names=two, world=world, counts_table=True).exchange \
        == "allgather"


@pytest.mark.parametrize("world", [1, 2, 8])
def test_one_rank_gathers_over_nccl(plan, world):
    p = plan(exchange="columns", transport="peer", world=world)
    if world == 1:
        assert (p.exchange, p.transport) == ("allgather", "nccl")
        # (one rank holds every column: a counts table is fine with exchange="columns")
        assert plan(exchange="columns", counts_table=True, world=world).exchange == "allgather"
    else:
        assert (p.exchange, p.transport) == ("columns", "peer")
        assert plan(exchange="allgather", transport="nccl", world=world).transport == "nccl"


@pytest.mark.parametrize("world", [1, 2, 8])
def test_density_takes_nccl(plan, world):
    p = plan(counter_names=["nucleotide-overlap", "nucleotide-density"], transport="peer", world=world,
             keep_samples=None, free_bytes=0)
    assert p.transport == "nccl"
    assert not p.matrix_free                # (density has no matrix-free mode: None keeps the matrix)


@pytest.mark.parametrize("world", [1, 2, 8])
def test_refusals(plan, world):
    if world > 1:
        with pytest.raises(ValueError, match="output_counts_pattern needs every column on rank 0"):
            plan(exchange="columns", counts_table=True, world=world)
    with pytest.raises(ValueError, match="exchange must be auto, allgather or columns"):
        plan(exchange="rows", world=world)
    with pytest.raises(ValueError, match="transport must be peer or nccl"):
        plan(transport="nvlink", world=world)
    with pytest.raises(ValueError, match="it needs keep_samples=True"):
        plan(keep_samples=False, counts_table=True, world=world)
    with pytest.raises(NotImplementedError, match="nucleotide-density has no matrix-free mode"):
        plan(keep_samples=False, counter_names=["nucleotide-density"], world=world)
    assert plan(keep_samples=False, world=world).matrix_free
    assert not plan(keep_samples=True, world=world, free_bytes=0).matrix_free


@pytest.mark.parametrize("world", [1, 2, 8])
@pytest.mark.parametrize("exchange", ["allgather", "columns"])
def test_matrix_bytes_of_this_rank(plan, world, exchange):
    """keep_samples=None: matrix-free exactly when the matrices this rank holds (4 * counters * S * its columns *
    tracks bytes) exceed the free memory; column-sharded, that is its own width of columns"""
    from gat_b200 import parallel
    S, A, T, C = 1000, 10, 3, 2
    names = ["nucleotide-overlap", "segment-overlap"]
    for rank in range(world):
        b, e = parallel.column_range(A, rank, world) if (exchange == "columns" and world > 1) else (0, A)
        need = 4 * C * S * (e - b) * T
        kw = dict(num_samples=S, n_annotations=A, n_tracks=T, counter_names=names, exchange=exchange,
                  keep_samples=None, rank=rank, world=world)
        assert not plan(free_bytes=need, **kw).matrix_free
        assert plan(free_bytes=need - 1, **kw).matrix_free


@pytest.mark.parametrize("world", [1, 2, 8])
@pytest.mark.parametrize("S,A", [(1001, 5), (7, 1), (4, 13)])
def test_row_and_column_ranges(plan, world, S, A):
    """the ranks' sample rows and columns tile [0, S) and [0, A) in rank order; all-gathered, every rank holds every
    column"""
    for exchange in ("allgather", "columns"):
        rows, cols = [], []
        for rank in range(world):
            p = plan(num_samples=S, n_annotations=A, exchange=exchange, rank=rank, world=world)
            rows.append(p.rows)
            cols.append(p.columns)
        assert rows[0][0] == 0 and rows[-1][1] == S
        assert all(rows[r][1] == rows[r + 1][0] for r in range(world - 1))
        if exchange == "columns" and world > 1:
            assert cols[0][0] == 0 and cols[-1][1] == A
            assert all(cols[r][1] == cols[r + 1][0] for r in range(world - 1))
        else:
            assert cols == [(0, A)] * world


# --------------------------------------------------------------------------------------------------- GPU
class Fold(object):
    def __init__(self, fold):
        self.fold = fold


def two_tracks():
    """the track "merged" and the track "outside", whose segments all lie beyond the end of the workspace: it has no
    placement unit"""
    from gat_b200 import synthetic
    from gat_b200.segmentlist import SegmentList
    segments, annotations, workspaces, _ = synthetic.make(
        n_segments=300, n_annotations=7, n_annotation_intervals=400, genome=[("chrA", 2000000), ("chrB", 1000000)])
    segments.add("outside", "chrA", SegmentList(array=np.array([[2100000, 2100500], [2500000, 2501000]],
                                                                dtype=np.uint32)))
    segments.normalize()
    workspace = synthetic.prepare(segments, annotations, workspaces)
    return segments, annotations, workspace


def run(segments, annotations, workspace, names, **kw):
    import gat_b200
    from gat_b200 import engine as Engine
    Engine.seed(5)
    return gat_b200.run(segments, annotations, workspace, Engine.SamplerAnnotator(),
                        [Engine.COUNTER_CLASSES[n]() for n in names], Engine.UnconditionalWorkspace(), **kw)


def phases_of(line):
    """the `# gat_b200.run phases:` line parsed as tools/run_cli_timed.py parses it -> (names in order, dict)"""
    m = re.search(r"# gat_b200.run phases: (.*)", line)
    parts = [x.rsplit(" ", 1) for x in m.group(1).split(", ")]
    return [k.strip() for k, _ in parts], dict((k.strip(), float(v[:-1])) for k, v in parts)


@pytest.mark.gpu
def test_track_without_units(tmp_path, monkeypatch, capfd):
    """every result of "outside" is the statistics of an all-zero uint32 matrix; the matrix and the matrix-free run
    agree and write the same samples files, none for "outside"; GATB_TIMING names each phase once"""
    import gat_b200
    from gat_b200 import TrackProblem
    segments, annotations, workspace = two_tracks()
    assert [len(TrackProblem(segments[t], workspace).unit_keys) > 0 for t in segments.tracks] == [True, False]
    atracks = list(annotations.tracks)
    folds = [0.01, 0.5, 1.0, 2.0, 1000.0, 0.25, 4.0]
    ref = [folds[i % len(folds)] for i in range(len(atracks))]
    reference = dict((t, dict((a, Fold(f)) for a, f in zip(atracks, ref))) for t in segments.tracks)
    S = 37
    monkeypatch.setenv("GATB_TIMING", "1")
    capfd.readouterr()
    out = {}
    for keep in (True, False):
        names = INTEGER_COUNTERS + (["nucleotide-density"] if keep else [])
        extra = dict(output_counts_pattern=str(tmp_path / "counts_%s.tsv")) if keep else {}
        out[keep] = run(segments, annotations, workspace, names, num_samples=S, keep_samples=keep, reference=reference,
                        output_samples_pattern=str(tmp_path / ("keep%i" % keep) / "samples_%s.bed"), **extra)
        got_names, seconds = phases_of(capfd.readouterr().err)
        assert len(got_names) == len(set(got_names)) == len(seconds)
        assert got_names == ["observed", "sampling"] + (["exchange"] if keep else []) + \
            ["overlap columns", "statistics+results"]
        zero = [r for r in out[keep] if r.track == "outside"]
        assert len(zero) == len(names) * len(atracks)
        for name in names:
            rs = [r for r in zero if r.counter == name]
            assert [r.annotation for r in rs] == atracks
            obs = np.array([r.observed for r in rs])
            want = gat_b200.getContext().column_stats(np.zeros((S, len(atracks)), dtype=np.uint32), obs,
                                                      pseudo_count=1.0, ref_fold=ref)
            for k in STATS:
                np.testing.assert_array_equal(np.array([getattr(r, k) for r in rs]), want[k], err_msg=(keep, name, k))
            for r in rs:
                assert r.nsamples == S
                if keep:
                    assert r.samples.dtype == np.float64 and np.array_equal(r.samples, np.zeros(S))
    # the statistics of both tracks agree between the modes (integer counters)
    keep_rows = [(r.track, r.annotation, r.counter, str(r)) for r in out[True] if r.counter in INTEGER_COUNTERS]
    assert keep_rows == [(r.track, r.annotation, r.counter, str(r)) for r in out[False]]
    for name in INTEGER_COUNTERS + ["nucleotide-density"]:
        with open(str(tmp_path / ("counts_%s.tsv" % name))) as f:
            rows = [line.rstrip("\n").split("\t") for line in f][1:]
        assert [row[3] for row in rows if row[0] == "outside"] == [",".join(["0"] * S)] * len(atracks)
    files = [sorted(os.listdir(str(tmp_path / ("keep%i" % keep)))) for keep in (True, False)]
    assert files[0] == files[1] == ["samples_merged.bed"]
    texts = [open(str(tmp_path / ("keep%i" % keep) / "samples_merged.bed")).read() for keep in (True, False)]
    assert texts[0] == texts[1] and texts[0].count("track name=") == S


@pytest.mark.gpu
@pytest.mark.parametrize("keep", [True, False])
def test_empty_workspace(keep):
    from gat_b200 import engine as Engine
    segments, annotations, _ = two_tracks()
    assert run(segments, annotations, Engine.IntervalDictionary(), INTEGER_COUNTERS, num_samples=20,
               keep_samples=keep) == []
