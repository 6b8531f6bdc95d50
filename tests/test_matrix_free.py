"""run(..., keep_samples=False): the statistics without the sample matrix (gat_b200/matrixfree.py, gatb_colacc_* in
include/gat_b200.h) are those of the matrix path, bit for bit.

The accumulator bodies run twice: on the GPU, and without one on the SIMT-emulated build of the same kernels
(tests/emu, as in tests/test_emu_parity.py)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))

STATS = ["expected", "stddev", "lower95", "upper95", "fold", "pvalue"]
BATCH = 4096                                # samples per internal batch of gatb_run


@pytest.fixture(scope="module")
def emu_ctx():
    import emu_context
    c = emu_context.context()
    yield c
    c.close()


def assert_identical(got, want, what=""):
    for k in STATS:
        assert np.array_equal(np.asarray(got[k]), np.asarray(want[k])), (what, k, got[k], want[k])


def planes_and_observed(rng, n_planes, S, A):
    """[n_planes][S][A] uint32 counts of different offsets and spreads (one constant column), and observed values
    below, at the bottom of, inside (integer: ties; not integer), at the top of and above every column's range"""
    mats = np.empty((n_planes, S, A), dtype=np.uint32)
    obs = np.empty((n_planes, A))
    for i in range(n_planes):
        base = rng.integers(0, 100000, A)
        spread = rng.integers(1, 400, A)
        spread[A // 2] = 1                  # a constant column
        mats[i] = base[None, :] + rng.integers(0, 1 << 30, (S, A)) % spread[None, :]
        m = mats[i]
        for a in range(A):
            c = m[:, a]
            obs[i, a] = [float(c.min()) - 3, float(c.min()), float(c[S // 2]), float(np.median(c)) + 0.5,
                         float(c.max()), float(c.max()) + 7, 0.0][a % 7]
    return mats, obs


class HostSlab(object):
    """the slab of the emulated build: "device" memory is host memory there"""

    def __init__(self, mats, chunk):
        self.mats = mats
        self.buf = np.zeros(mats.shape[0] * chunk * mats.shape[2], dtype=np.uint32)

    def __call__(self, r0, n):
        P, _, A = self.mats.shape
        self.buf[:P * n * A] = self.mats[:, r0:r0 + n].reshape(-1)
        return self.buf.ctypes.data


class DeviceSlab(object):
    def __init__(self, mats, chunk):
        import torch
        self.mats = torch.from_numpy(mats.view(np.int32)).cuda()
        self.buf = torch.zeros(mats.shape[0] * chunk * mats.shape[2], dtype=torch.int32, device="cuda")

    def __call__(self, r0, n):
        P, _, A = self.mats.shape
        self.buf[:P * n * A].copy_(self.mats[:, r0:r0 + n].reshape(-1))
        return self.buf.data_ptr()


def check_stream_statistics(ctx, slab_class, S, A, chunk, with_ref, pilot_window=None, seed=0):
    """slabs of `chunk` rows through the accumulators == gatb_column_stats on the whole matrix"""
    from gat_b200 import matrixfree
    rng = np.random.default_rng(seed)
    mats, obs = planes_and_observed(rng, 2, S, A)
    ref = rng.choice([0.01, 0.5, 1.0, 3.0, 1000.0], A) if with_ref else None
    want = [ctx.column_stats(mats[i], obs[i], pseudo_count=1.0, ref_fold=ref) for i in range(2)]
    reruns = matrixfree.info["reruns"]
    old = matrixfree.PILOT_WINDOW
    matrixfree.PILOT_WINDOW = pilot_window
    try:
        got = matrixfree.stream_statistics(ctx, slab_class(mats, chunk), [(obs[i], ref) for i in range(2)], S, S, A,
                                           chunk, pseudo_count=1.0, budget_bytes=1 << 30)
    finally:
        matrixfree.PILOT_WINDOW = old
    for i in range(2):
        assert_identical(got[i], want[i], (S, A, chunk, i))
    return matrixfree.info["reruns"] - reruns


def check_merge_of_two_ranks(ctx, slab_class, S, A):
    """two accumulators with half the rows each, one state merged into the other (128-bit carries included) ==
    gatb_column_stats on the whole matrix"""
    from gat_b200 import device
    rng = np.random.default_rng(3)
    mats, obs = planes_and_observed(rng, 1, S, A)
    mats[0, :, 0] = 0xffffffff - rng.integers(0, 3, S).astype(np.uint32)   # sums of squares beyond 2^64
    obs[0, 0] = 4294967294.0
    want = ctx.column_stats(mats[0], obs[0])
    lo = mats[0].min(axis=0)
    width = mats[0].max(axis=0) - lo + 1
    half = S // 2
    accs = []
    for r0, r1 in ((0, half), (half, S)):
        acc = device.ColumnAccumulator(ctx, A, S, obs[0])
        acc.set_windows(lo, width)
        slab = slab_class(mats[:, r0:r1], r1 - r0)
        acc.add(slab(0, r1 - r0), r1 - r0)
        accs.append(acc)
    with pytest.raises(Exception):
        accs[0].finish()                    # (half of the samples)
    accs[0].merge(accs[1].state())
    got, missed = accs[0].finish()
    assert not missed.any()
    assert_identical(got, want)
    for a in accs:
        a.close()


# ---------------------------------------------------------------------------------------------- without a GPU
def test_decision_of_the_default_mode():
    from gat_b200.matrixfree import use_matrix_free
    assert use_matrix_free(None, False, False, 8 << 30, 4 << 30)
    assert not use_matrix_free(None, False, False, 4 << 30, 8 << 30)
    assert not use_matrix_free(None, True, False, 8 << 30, 4 << 30)        # a counts table needs the samples
    assert not use_matrix_free(None, False, True, 8 << 30, 4 << 30)        # density: float64, matrix only
    assert use_matrix_free(False, False, False, 0, 1 << 40)
    assert not use_matrix_free(True, False, False, 1 << 40, 0)
    with pytest.raises(ValueError):
        use_matrix_free(False, True, False, 0, 0)
    with pytest.raises(NotImplementedError):
        use_matrix_free(False, False, True, 0, 0)


@pytest.mark.parametrize("S,A,chunk,with_ref", [(1, 9, 1, False), (20, 9, 7, True), (21, 9, 21, False),
                                                (97, 30, 40, True), (64, 2051, 25, False)])
def test_accumulator_on_the_emulated_kernels(emu_ctx, S, A, chunk, with_ref):
    """A = 2051: wider than a ring stage of the streamed pass, the column-tiled pass 1 accumulates"""
    check_stream_statistics(emu_ctx, HostSlab, S, A, chunk, with_ref)


def test_window_miss_on_the_emulated_kernels(emu_ctx):
    assert check_stream_statistics(emu_ctx, HostSlab, 90, 14, 31, True, pilot_window=1) == 1


def test_merge_of_two_ranks_on_the_emulated_kernels(emu_ctx):
    check_merge_of_two_ranks(emu_ctx, HostSlab, 41, 9)


# --------------------------------------------------------------------------------------------------- GPU
@pytest.fixture
def gpu_ctx(ctx):
    import torch
    ctx.set_stream(torch.cuda.current_stream().cuda_stream or 1)
    yield ctx
    torch.cuda.synchronize()
    ctx.set_stream(None)


@pytest.mark.gpu
@pytest.mark.parametrize("S,A,chunk,with_ref", [(1, 9, 1, False), (20, 1000, 7, True), (4097, 1000, 1500, False),
                                                (3 * BATCH + 5, 333, 4096, True), (3000, 2051, 1024, True)])
def test_accumulator_matches_column_stats(gpu_ctx, S, A, chunk, with_ref):
    check_stream_statistics(gpu_ctx, DeviceSlab, S, A, chunk, with_ref)


@pytest.mark.gpu
def test_accumulator_window_miss(gpu_ctx):
    assert check_stream_statistics(gpu_ctx, DeviceSlab, 5000, 200, 1024, False, pilot_window=1) == 1


@pytest.mark.gpu
def test_accumulator_merge_of_two_ranks(gpu_ctx):
    check_merge_of_two_ranks(gpu_ctx, DeviceSlab, 4001, 300)


class Fold(object):
    def __init__(self, fold):
        self.fold = fold


def problem(isochores):
    from gat_b200 import synthetic
    segments, annotations, workspaces, iso = synthetic.make(
        n_segments=300, n_annotations=7, n_annotation_intervals=400, isochores=isochores,
        genome=[("chrA", 2000000), ("chrB", 1000000)], isochore_tile=50000, n_isochores=3)
    workspace = synthetic.prepare(segments, annotations, workspaces, iso)
    return segments, annotations, workspace


INTEGER_COUNTERS = ["nucleotide-overlap", "segment-overlap", "segment-midoverlap", "annotation-overlap",
                    "annotation-midoverlap"]


def run_both(segments, annotations, workspace, make_sampler, S, reference=None, counters=INTEGER_COUNTERS, **kw):
    import gat_b200
    from gat_b200 import engine as Engine
    out = []
    for keep in (True, False):
        Engine.seed(11)
        out.append(gat_b200.run(segments, annotations, workspace, make_sampler(),
                                [Engine.COUNTER_CLASSES[n]() for n in counters], Engine.UnconditionalWorkspace(),
                                num_samples=S, reference=reference, keep_samples=keep, **kw))
    return out


def assert_runs_identical(a, b):
    assert len(a) == len(b) and len(a) > 0
    for x, y in zip(a, b):
        assert (x.track, x.annotation, x.counter, x.observed) == (y.track, y.annotation, y.counter, y.observed)
        for k in ("expected", "stddev", "lower95", "upper95", "fold", "pvalue", "qvalue", "nsamples"):
            assert getattr(x, k) == getattr(y, k), (x.counter, x.annotation, k, getattr(x, k), getattr(y, k))
        assert str(x) == str(y)


SAMPLERS = {
    "annotator": lambda: __import__("gat_b200").SamplerAnnotator(),
    "segments": lambda: __import__("gat_b200").SamplerSegments(),
    "shift": lambda: __import__("gat_b200").SamplerShift(radius=2),
}


@pytest.mark.gpu
@pytest.mark.parametrize("sampler,isochores,S", [("annotator", False, S) for S in (1, 19, 20, 21, 4095, 4097, 3 * BATCH + 5)]
                         + [("annotator", True, 4097), ("segments", True, 21), ("segments", True, 4097),
                            ("shift", False, 4097), ("shift", True, 20)])
@pytest.mark.parametrize("with_ref", [False, True])
def test_run_without_the_matrix_is_bit_identical(monkeypatch, sampler, isochores, S, with_ref):
    """all five integer counters at once; slabs of 1500 rows (neither a batch nor a divisor of S); with a
    reference, folds of 0.01 and 1000 put the observed value below and above the sampled range"""
    from gat_b200 import matrixfree
    segments, annotations, workspace = problem(isochores)
    atracks = list(annotations.tracks)
    reference = None
    if with_ref:
        folds = [0.01, 0.5, 1.0, 2.0, 1000.0, 0.25, 4.0]
        reference = dict((t, dict((a, Fold(folds[i % len(folds)])) for i, a in enumerate(atracks)))
                         for t in segments.tracks)
    monkeypatch.setattr(matrixfree, "SLAB_BYTES", 4 * len(INTEGER_COUNTERS) * len(atracks) * 1500)
    keep, free = run_both(segments, annotations, workspace, SAMPLERS[sampler], S, reference)
    assert_runs_identical(keep, free)


@pytest.mark.gpu
def test_run_window_miss_reruns_and_stays_identical(monkeypatch):
    from gat_b200 import matrixfree
    segments, annotations, workspace = problem(False)
    monkeypatch.setattr(matrixfree, "PILOT_WINDOW", 1)
    monkeypatch.setattr(matrixfree, "SLAB_BYTES", 4 * len(INTEGER_COUNTERS) * 7 * 1000)
    keep, free = run_both(segments, annotations, workspace, SAMPLERS["annotator"], 5000)
    assert matrixfree.info["reruns"] >= 1
    assert_runs_identical(keep, free)


@pytest.mark.gpu
def test_run_refusals_and_results_without_samples(tmp_path):
    import gat_b200
    from gat_b200 import engine as Engine
    segments, annotations, workspace = problem(False)

    def go(counters, **kw):
        Engine.seed(3)
        return gat_b200.run(segments, annotations, workspace, Engine.SamplerAnnotator(),
                            [Engine.COUNTER_CLASSES[n]() for n in counters], Engine.UnconditionalWorkspace(),
                            num_samples=50, **kw)
    with pytest.raises(ValueError):
        go(["nucleotide-overlap"], keep_samples=False, output_counts_pattern=str(tmp_path / "c_%s.tsv"))
    with pytest.raises(NotImplementedError):
        go(["nucleotide-density"], keep_samples=False)
    res = go(["segment-overlap"], keep_samples=False)
    ref = go(["segment-overlap"])                   # default: fits, the matrix path
    assert ref[0].samples.shape == (50,)
    for r in res:
        assert r.nsamples == 50
        for f in (lambda: r.samples, lambda: r.getSample(0), lambda: r.getEmpiricalPValue(r.observed)):
            with pytest.raises(RuntimeError, match="keep_samples=True"):
                f()
    Engine.updateQValues(res, method="BH")
    Engine.updateQValues(ref, method="BH")
    Engine.updatePValues(res, "norm")
    Engine.updatePValues(ref, "norm")
    assert [str(x) for x in res] == [str(x) for x in ref]


@pytest.mark.gpu
def test_run_memory_does_not_grow_with_the_samples():
    """A = 1000 annotation tracks: the device memory a matrix-free run adds (the largest drop of free memory,
    cudaMemGetInfo, after every slab, from just before the run) is the same at S = 2e5 (already one full slab of
    134 217 rows) and at S = 2e6, where the matrix would be 8 GB, and a small fraction of that matrix.  A warm-up run
    first fills the library's pools (annotation index, batch buffers: what the matrix path needs as well); torch's
    cached blocks are released before each measured run (they are kept per stream, and every run has its own)."""
    import torch
    import gat_b200
    from gat_b200 import engine as Engine, matrixfree, synthetic
    segments, annotations, workspaces, _ = synthetic.make(n_segments=500, n_annotations=1000, n_annotation_intervals=20000)
    workspace = synthetic.prepare(segments, annotations, workspaces)
    A = len(list(annotations.tracks))
    orig = matrixfree.stream_statistics

    def run(S):
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        free0 = torch.cuda.mem_get_info()[0]
        peak = [0]

        def spy(ctx, produce, *args, **kw):
            def produce_and_measure(r0, n):
                ptr = produce(r0, n)
                torch.cuda.synchronize()
                peak[0] = max(peak[0], free0 - torch.cuda.mem_get_info()[0])
                return ptr
            return orig(ctx, produce_and_measure, *args, **kw)
        Engine.seed(1)
        try:
            matrixfree.stream_statistics = spy
            res = gat_b200.run(segments, annotations, workspace, Engine.SamplerAnnotator(),
                               [Engine.CounterNucleotideOverlap()], Engine.UnconditionalWorkspace(),
                               num_samples=S, keep_samples=False)
        finally:
            matrixfree.stream_statistics = orig
        assert len(res) == A and all(r.nsamples == S for r in res)
        return peak[0]
    run(20000)
    small, big = run(200000), run(2000000)
    matrix = 4 * 2000000 * A
    print("matrix %i B; device memory added at S = 2e5: %i B, at S = 2e6: %i B; histogram arena %i B, %i rows per slab"
          % (matrix, small, big, matrixfree.info["arena_bytes"], matrixfree.info["chunk_rows"]))
    assert 0 < big <= small + (64 << 20)
    assert big < matrix // 8
    assert matrixfree.info["arena_bytes"] < matrix // 64


@pytest.mark.gpu
def test_multirank_matrix_free_equals_single_rank_matrix():
    """2 ranks in the matrix-free mode give the 1-rank matrix-mode results exactly (tools/multirank_check.py
    --keep-samples 0).  Needs two GPUs: skipped on a one-GPU box."""
    import json
    import subprocess
    import torch
    from tests.test_parallel_gloo import free_port
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", str(free_port()),
                          os.path.join(ROOT, "tools", "multirank_check.py"), "--samples", "2001", "--tracks", "12",
                          "--keep-samples", "0"],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout + out.stderr
    line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
    assert json.loads(line)["ok"]
