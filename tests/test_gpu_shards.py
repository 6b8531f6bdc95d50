"""Sharded runs on the GPU: shard jobs (gat_b200.runShard, `gat_b200.cli --sample-range`) merged with mergeShards
(`python -m gat_b200.shards`) give the results of one run() over all samples, compared with ==."""
import os
import random
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BATCH = 4096                                # samples per internal batch of gatb_run
INTEGER_COUNTERS = ["nucleotide-overlap", "segment-overlap", "segment-midoverlap", "annotation-overlap",
                    "annotation-midoverlap"]
STATS = ["expected", "stddev", "lower95", "upper95", "fold", "pvalue"]
SAMPLERS = {
    "annotator": lambda: __import__("gat_b200").SamplerAnnotator(),
    "segments": lambda: __import__("gat_b200").SamplerSegments(),
    "shift": lambda: __import__("gat_b200").SamplerShift(radius=2),
}


class Fold(object):
    def __init__(self, fold):
        self.fold = fold


def problem(isochores):
    """7 annotation tracks; without isochores also the track "outside", whose segments all lie beyond the end of the
    workspace (no placement unit: every sample counts zero)"""
    from gat_b200 import synthetic
    from gat_b200.segmentlist import SegmentList
    segments, annotations, workspaces, iso = synthetic.make(
        n_segments=300, n_annotations=7, n_annotation_intervals=400, isochores=isochores,
        genome=[("chrA", 2000000), ("chrB", 1000000)], isochore_tile=50000, n_isochores=3)
    if not isochores:
        segments.add("outside", "chrA", SegmentList(array=np.array([[2100000, 2100500], [2500000, 2501000]],
                                                                    dtype=np.uint32)))
        segments.normalize()
    workspace = synthetic.prepare(segments, annotations, workspaces, iso)
    return segments, annotations, workspace


def splits(S, k):
    """k uneven ranges that tile [0, S), or None"""
    cuts = {1: [0, S], 2: [0, min(BATCH, S - 1), S], 3: [0, 1, S - 1, S],
            5: [0, 1, S // 3, S // 2, S - 1, S]}[k]
    if any(b >= e for b, e in zip(cuts[:-1], cuts[1:])):
        return None
    return list(zip(cuts[:-1], cuts[1:]))


def assert_runs_identical(a, b):
    assert len(a) == len(b) and len(a) > 0
    for x, y in zip(a, b):
        assert (x.track, x.annotation, x.counter, x.observed) == (y.track, y.annotation, y.counter, y.observed)
        for k in STATS + ["qvalue", "nsamples"]:
            assert getattr(x, k) == getattr(y, k), (x.track, x.counter, x.annotation, k, getattr(x, k), getattr(y, k))
        assert str(x) == str(y)


def run_whole(inputs, make_sampler, S, reference=None, counters=INTEGER_COUNTERS):
    import gat_b200
    from gat_b200 import engine as Engine
    segments, annotations, workspace = inputs
    Engine.seed(11)
    return gat_b200.run(segments, annotations, workspace, make_sampler(), [Engine.COUNTER_CLASSES[n]() for n in counters],
                        Engine.UnconditionalWorkspace(), num_samples=S, reference=reference, keep_samples=True)


def run_shards(tmp_path, tag, inputs, make_sampler, S, ranges, reference=None, counters=INTEGER_COUNTERS):
    """one shard job per range -> the files, shuffled"""
    import gat_b200
    from gat_b200 import engine as Engine
    segments, annotations, workspace = inputs
    files = []
    for i, r in enumerate(ranges):
        Engine.seed(11)
        f = str(tmp_path / ("%s_%i.npz" % (tag, i)))
        assert gat_b200.runShard(segments, annotations, workspace, make_sampler(),
                                 [Engine.COUNTER_CLASSES[n]() for n in counters], Engine.UnconditionalWorkspace(), r, f,
                                 num_samples=S, reference=reference) is None
        files.append(f)
    random.Random(S + len(ranges)).shuffle(files)
    return files


@pytest.mark.gpu
@pytest.mark.parametrize("sampler,isochores,S", [("annotator", False, S) for S in (1, 20, 4097, 3 * BATCH + 5)]
                         + [("annotator", True, 4097), ("segments", True, 20), ("segments", True, 4097),
                            ("shift", False, 4097), ("shift", True, 20)])
@pytest.mark.parametrize("with_ref", [False, True])
def test_merged_shards_equal_the_run(tmp_path, monkeypatch, sampler, isochores, S, with_ref):
    """1, 2, 3 and 5 shards, uneven and shuffled, all five integer counters; slabs of 1500 rows, so that the larger
    shards sample their histogram pass again and the smaller ones read it from the slab"""
    import gat_b200
    from gat_b200 import matrixfree
    inputs = problem(isochores)
    atracks = list(inputs[1].tracks)
    reference = None
    if with_ref:
        folds = [0.01, 0.5, 1.0, 2.0, 1000.0, 0.25, 4.0]
        reference = dict((t, dict((a, Fold(folds[i % len(folds)])) for i, a in enumerate(atracks)))
                         for t in inputs[0].tracks)
    monkeypatch.setattr(matrixfree, "SLAB_BYTES", 4 * len(INTEGER_COUNTERS) * len(atracks) * 1500)
    whole = run_whole(inputs, SAMPLERS[sampler], S, reference)
    if not isochores:
        assert "outside" in set(r.track for r in whole)
    for k in (1, 2, 3, 5):
        ranges = splits(S, k)
        if ranges is None:
            continue
        merged = gat_b200.mergeShards(run_shards(tmp_path, "k%i" % k, inputs, SAMPLERS[sampler], S, ranges, reference))
        assert_runs_identical(whole, merged)
        for r in merged[:3]:
            for f in (lambda: r.samples, lambda: r.getSample(0), lambda: r.getEmpiricalPValue(r.observed)):
                with pytest.raises(RuntimeError, match="keep_samples=True"):
                    f()


@pytest.mark.gpu
def test_shard_larger_than_its_slab_samples_pass_two_again(tmp_path, monkeypatch):
    import gat_b200
    from gat_b200 import engine as Engine, matrixfree
    inputs = problem(False)
    S = 5000
    whole = run_whole(inputs, SAMPLERS["annotator"], S)
    monkeypatch.setattr(matrixfree, "SLAB_BYTES", 4 * len(INTEGER_COUNTERS) * 7 * 1000)
    files = run_shards(tmp_path, "big", inputs, SAMPLERS["annotator"], S, [(0, 4000)])
    assert matrixfree.info["chunk_rows"] == 1000
    assert matrixfree.info["reruns"] == 2                 # (both tracks of the job: 4000 rows in slabs of 1000)
    files += run_shards(tmp_path, "fits", inputs, SAMPLERS["annotator"], S, [(4000, 5000)])
    assert matrixfree.info["reruns"] == 0                 # (1000 rows: pass 2 reads the slab still in the buffer)
    merged = gat_b200.mergeShards(files)
    assert_runs_identical(whole, merged)
    # q-values and the normal p-values work on merged results as on run()'s
    Engine.updateQValues(whole, method="BH")
    Engine.updateQValues(merged, method="BH")
    Engine.updatePValues(whole, "norm")
    Engine.updatePValues(merged, "norm")
    assert [str(x) for x in whole] == [str(x) for x in merged]


@pytest.mark.gpu
def test_shard_refusals(tmp_path):
    import gat_b200
    from gat_b200 import engine as Engine
    segments, annotations, workspace = problem(False)

    def go(counters=("nucleotide-overlap",), seeded=True, rng=(0, 10), **kw):
        if seeded:
            Engine.seed(3)
        else:
            Engine._rng_state.update(seed=None, calls=0)
        return gat_b200.runShard(segments, annotations, workspace, Engine.SamplerAnnotator(),
                                 [Engine.COUNTER_CLASSES[n]() for n in counters], Engine.UnconditionalWorkspace(), rng,
                                 str(tmp_path / "x.npz"), num_samples=20, **kw)
    with pytest.raises(ValueError, match="seeded"):
        go(seeded=False)
    with pytest.raises(ValueError, match="keep_samples=True"):
        go(keep_samples=True)
    with pytest.raises(ValueError, match="output_counts_pattern"):
        go(output_counts_pattern=str(tmp_path / "c_%s.tsv"))
    with pytest.raises(ValueError, match="sample_range"):
        go(rng=(10, 21))
    with pytest.raises(NotImplementedError, match="nucleotide-density"):
        go(counters=("nucleotide-density",))
    assert not os.path.exists(str(tmp_path / "x.npz"))
    go()
    # shards of another seed or other inputs do not merge
    first = str(tmp_path / "first.npz")
    os.rename(str(tmp_path / "x.npz"), first)
    Engine.seed(4)
    gat_b200.runShard(segments, annotations, workspace, Engine.SamplerAnnotator(), [Engine.CounterNucleotideOverlap()],
                      Engine.UnconditionalWorkspace(), (10, 20), str(tmp_path / "seed.npz"), num_samples=20)
    with pytest.raises(ValueError, match="seed"):
        gat_b200.mergeShards([first, str(tmp_path / "seed.npz")])
    Engine.seed(3)
    gat_b200.runShard(segments, annotations, workspace, Engine.SamplerShift(), [Engine.CounterNucleotideOverlap()],
                      Engine.UnconditionalWorkspace(), (10, 20), str(tmp_path / "shift.npz"), num_samples=20)
    with pytest.raises(ValueError, match="digest"):
        gat_b200.mergeShards([first, str(tmp_path / "shift.npz")])


@pytest.mark.gpu
def test_sum_of_squares_past_two_to_the_64_through_shard_files(ctx, tmp_path):
    """values near 2^32: the shards' 128-bit sums of squares carry when they are added, as in test_matrix_free's
    two-accumulator merge"""
    import torch
    from gat_b200 import matrixfree, shards
    from tests.test_shards import _file
    ctx.set_stream(torch.cuda.current_stream().cuda_stream or 1)
    try:
        rng = np.random.default_rng(3)
        S, A = 4001, 300
        mats = (rng.integers(0, 100000, A)[None, None, :] + rng.integers(0, 400, (2, S, A))).astype(np.uint32)
        mats[0, :, 0] = 0xffffffff - rng.integers(0, 3, S).astype(np.uint32)
        obs = np.stack([mats[i, S // 2].astype(np.float64) for i in range(2)])
        obs[0, 0] = 4294967294.0
        want = [ctx.column_stats(mats[i], obs[i]) for i in range(2)]
        dev = torch.from_numpy(mats.view(np.int32)).cuda()
        files = []
        for k, (b, e) in enumerate([(0, 1), (1, 2000), (2000, S)]):
            buf = torch.zeros(2 * 1024 * A, dtype=torch.int32, device="cuda")

            def produce(r0, n, b=b, buf=buf):
                buf[:2 * n * A].copy_(dev[:, b + r0:b + r0 + n].reshape(-1))
                return buf.data_ptr()
            states = matrixfree.shard_states(ctx, produce, [(obs[i], None) for i in range(2)], S, e - b, A, 1024)
            files.append(_file(tmp_path / ("s%i.npz" % k), S, (b, e), obs, None, states))
        sq = [shards.Shard(f).state(0, 0)["moments"] for f in files]
        total = sum((int(m[4][0]) << 64) + int(m[3][0]) for m in sq)
        assert total >= 1 << 64 and sum(int(m[3][0]) for m in sq) >= 1 << 64      # (the low words carry)
        got = shards._merge(shards.readShards(files), ctx)
        for i, name in enumerate(["nucleotide-overlap", "segment-overlap"]):
            for k in STATS:
                assert np.array_equal(np.array([getattr(r, k) for r in got if r.counter == name]), want[i][k]), (i, k)
    finally:
        torch.cuda.synchronize()
        ctx.set_stream(None)


# ----------------------------------------------------------------------------------------------- command line
def write_inputs(tmp_path, isochores):
    from gat_b200 import synthetic
    segments, annotations, workspaces, iso = synthetic.make(
        n_segments=300, n_annotations=7, n_annotation_intervals=400, isochores=isochores,
        genome=[("chrA", 2000000), ("chrB", 1000000)], isochore_tile=50000, n_isochores=3)
    args = []
    for name, coll, tracks in (("segments", segments, False), ("annotations", annotations, True),
                               ("workspace", workspaces, False)) + ((("isochore-file", iso, True),) if isochores else ()):
        path = str(tmp_path / (name + ".bed"))
        synthetic.write_bed(coll, path, with_tracks=tracks)
        args.append("--%s=%s" % (name, path))
    return args


def cli_tables(tmp_path, tag, args, counters):
    """the table files a run wrote: stdout for one counter, one per counter else"""
    if len(counters) == 1:
        return [open(str(tmp_path / (tag + ".tsv"))).read()]
    return [open(str(tmp_path / ("%s_%s.tsv" % (tag, c)))).read() for c in counters]


def output_args(tmp_path, tag):
    return ["--stdout=" + str(tmp_path / (tag + ".tsv")), "--output-tables-pattern=" + str(tmp_path / (tag + "_%s.tsv"))]


@pytest.mark.gpu
@pytest.mark.parametrize("isochores,counters,extra", [
    (False, ["nucleotide-overlap"], []),
    (True, ["nucleotide-overlap", "segment-overlap"], ["-q", "storey"])])
def test_cli_shards_print_the_table_of_one_run(tmp_path, isochores, counters, extra):
    from gat_b200 import cli, shards
    S = 300
    common = write_inputs(tmp_path, isochores) + ["--counter=" + c for c in counters] + \
        ["--num-samples=%i" % S, "--random-seed=7", "-v", "0"]
    assert cli.main(["gat-run"] + common + extra + output_args(tmp_path, "whole")) == 0
    files = []
    for i, (b, e) in enumerate([(250, 300), (0, 100), (100, 250)]):
        f = str(tmp_path / ("part%i.npz" % i))
        assert cli.main(["gat-run"] + common + ["--sample-range=%i:%i" % (b, e), "--output-shard=" + f,
                                                "--stdout=" + str(tmp_path / "shard_stdout.txt")]) == 0
        assert open(str(tmp_path / "shard_stdout.txt")).read() == ""           # (a shard job prints no table)
        files.append(f)
    assert shards.main(["gat-merge"] + extra + output_args(tmp_path, "merged") + files) == 0
    want, got = cli_tables(tmp_path, "whole", common, counters), cli_tables(tmp_path, "merged", common, counters)
    assert len(want[0].splitlines()) > 1 and got == want
    with pytest.raises(ValueError, match="--random-seed"):
        cli.main(["gat-run"] + [a for a in common if not a.startswith("--random-seed")] +
                 ["--sample-range=0:10", "--output-shard=" + str(tmp_path / "x.npz")])


@pytest.mark.gpu
def test_two_rank_shard_and_one_rank_shard_merge_to_the_one_rank_run(tmp_path):
    """a shard job on two ranks (torch.distributed.run) plus a one-rank shard job, merged, print the table of the
    one-rank run.  Needs two GPUs: skipped on a one-GPU box."""
    import torch
    from gat_b200 import cli, shards
    from tests.test_parallel_gloo import free_port
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    S = 2001
    common = write_inputs(tmp_path, False) + ["--counter=nucleotide-overlap", "--counter=segment-overlap",
                                              "--num-samples=%i" % S, "--random-seed=5", "-v", "0"]
    assert cli.main(["gat-run"] + common + output_args(tmp_path, "whole")) == 0
    two = str(tmp_path / "two.npz")
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", str(free_port()), "-m", "gat_b200.cli"]
                         + common + ["--sample-range=0:1500", "--output-shard=" + two],
                         capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stdout + out.stderr
    one = str(tmp_path / "one.npz")
    assert cli.main(["gat-run"] + common + ["--sample-range=1500:%i" % S, "--output-shard=" + one]) == 0
    assert shards.main(["gat-merge"] + output_args(tmp_path, "merged") + [one, two]) == 0
    counters = ["nucleotide-overlap", "segment-overlap"]
    assert cli_tables(tmp_path, "merged", common, counters) == cli_tables(tmp_path, "whole", common, counters)
