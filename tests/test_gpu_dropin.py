"""The drop-in claim, exercised (VERDICT r1 #9): the binding of INTEGRATION.md section 2 (integration/_b200.py, ctypes
against libgat_b200.so, nothing of the gat_b200 package), installed as UnconditionalSampler.sample and
Engine.computeCounts, reproduces the reference's own runs.  The binding reads the reference's containers through
their pickled segment buffers; the tests hand it containers of the same shape (_RefCollection below, over the
golden inputs) and call the two entry points the way the reference's gat.run() does (_run below), so they need
no copy of the reference.  Inputs: the reference's golden run (test/data, prepared intervals in
tests/golden/observed_testdata.npz) and the tutorial (tests/golden/observed_tutorial.npz), plus the small runs
whose sampled distributions the reference produced itself (tests/golden/distribution.npz).

  observed            bit-exact against the reference's own numbers (28 golden values, 20183)
  expected / fold     within Monte-Carlo error of the reference's published table and of its own samples
  statistics          of the binding's samples by the CPU oracle's restatement of the reference's AnnotatorResult
  same matrix         the binding-driven run and gat_b200.run() see identical sample columns for one seed
"""
import importlib.util
import os
import types

import numpy as np
import pytest

from tests import golden_util as G

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _RefList(object):
    """a reference SegmentList as the binding reads it: len, isEmpty and __reduce__, whose sixth argument is the
    buffer of raw {uint32 start, end} pairs (gat/SegmentList.pyx:262-337)"""

    def __init__(self, array=None):
        self.array = np.ascontiguousarray(np.zeros((0, 2)) if array is None else array, dtype=np.uint32).reshape(-1, 2)

    def __len__(self):
        return len(self.array)

    @property
    def isEmpty(self):
        return len(self.array) == 0

    def __reduce__(self):
        n = len(self.array)
        return (_RefList, (n, n, 1, 10000, None, self.array.tobytes()))


class _RefDictionary(dict):
    """a reference IntervalDictionary (key -> SegmentList) over a gat_b200 one; clone / fromIsochores / sum are the
    gat_b200 ones, which restate the reference's"""

    def __init__(self, source):
        dict.__init__(self)
        self.source = source
        self._wrap()

    def _wrap(self):
        self.clear()
        self.update((k, _RefList(s.asarray())) for k, s in self.source.items())

    def clone(self):
        return type(self)(self.source.clone())

    def fromIsochores(self):
        self.source.fromIsochores()
        self._wrap()

    def sum(self):
        return self.source.sum()


class _RefCollection(_RefDictionary):
    """a reference IntervalCollection (track -> IntervalDictionary) over a gat_b200 one"""

    def _wrap(self):
        self.clear()
        self.update((t, _RefDictionary(d)) for t, d in self.source.items())

    @property
    def tracks(self):
        return list(self.keys())


def _reference_entry_points():
    """the two entry points of the reference the binding replaces, as install() finds them"""
    class UnconditionalSampler(object):
        def __init__(self, num_samples, sampler, workspace_generator):
            self.num_samples, self.sampler, self.workspace_generator = num_samples, sampler, workspace_generator

        def sample(self, *args):
            raise AssertionError("the binding is not installed")

    def computeCounts(*args, **kwargs):
        raise AssertionError("the binding is not installed")

    return types.SimpleNamespace(UnconditionalSampler=UnconditionalSampler,
                                 Engine=types.SimpleNamespace(computeCounts=computeCounts))


@pytest.fixture(scope="module")
def ref():
    """(reference entry points with the binding installed, the binding module)"""
    gat = _reference_entry_points()
    spec = importlib.util.spec_from_file_location("gat_b200_binding", os.path.join(ROOT, "integration", "_b200.py"))
    binding = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(binding)
    uninstall = binding.install(gat)
    yield gat, binding
    uninstall()


def _run(gat, segments, annotations, workspace, counter_names, num_samples):
    """what the reference's gat.run() asks of the two replaced entry points (gat/__init__.py:932-1000): the
    observed counts of every counter, then UnconditionalSampler.sample once per segment track
    -> {(track, annotation, counter): (observed, samples)}"""
    from gat_b200 import engine as Engine
    rs, ra, rw = _RefCollection(segments), _RefCollection(annotations), _RefDictionary(workspace)
    generator = Engine.UnconditionalWorkspace()
    counters = [Engine.COUNTER_CLASSES[n]() for n in counter_names]
    observed = [gat.Engine.computeCounts(c, sum, rs, ra, rw, generator) for c in counters]
    outer = gat.UnconditionalSampler(num_samples, Engine.SamplerAnnotator(bucket_size=1, nbuckets=100000), generator)
    out = {}
    for track in rs.tracks:
        counts = outer.sample(track, None, counters, rs[track], ra, rw, {})
        for ci, c in enumerate(counters):
            for a in ra.tracks:
                out[(track, a, c.name)] = (observed[ci][track][a], np.asarray(counts[ci][a], dtype=np.float64))
    return out


def test_reference_run_on_the_library_golden_testdata(ctx, ref, oracle):
    """the reference's own golden run (test/data/output_single.tsv): 28 observed values bit-exact through
    gatb_count_lists, 200 samples per track on top of gatb_run"""
    gat, binding = ref
    z, meta = G.load_npz("observed_testdata")
    segments = G.collection(z, "segments", meta["segments"], coded=True)
    annotations = G.collection(z, "annotations", meta["annotations"], coded=True)
    workspace = G.dictionary(z, "workspace", meta["workspace"], coded=True)
    binding.seed(11)
    results = _run(gat, segments, annotations, workspace, ["nucleotide-overlap"], 200)
    got = dict(("%s|%s" % (t, a), v) for (t, a, _), v in results.items())
    assert len(meta["golden"]) == 28 and sorted(got) == sorted(meta["golden"])
    for key, observed in meta["golden"].items():
        obs, samples = got[key]
        assert isinstance(obs, int) and obs == int(observed), key
        st = oracle.enrichment_statistics(obs, samples)
        assert len(samples) == 200 and 0 < st.pvalue <= 1 and st.expected >= 0


def test_reference_run_on_the_library_tutorial(ctx, ref, oracle):
    """doc/tutorialIntervalOverlap.rst: observed 20183 bit-exact; expected / stddev / fold agree with the published
    1000-sample table (expected 246.565, stddev 105.59, fold 81.53) within Monte-Carlo error"""
    from gat_b200 import engine as Engine
    gat, binding = ref
    z, meta = G.load_npz("observed_tutorial")
    segments = G.collection(z, "segments", meta["segments"], coded=True)
    annotations = G.collection(z, "annotations", meta["annotations"], coded=True)
    workspace = G.dictionary(z, "workspace", meta["workspace"], coded=True)
    binding.seed(3)
    results = _run(gat, segments, annotations, workspace, ["nucleotide-overlap"], 500)
    assert len(results) == 1
    (track, annotation, counter), (obs, samples) = list(results.items())[0]
    r, pub = oracle.enrichment_statistics(obs, samples), meta["published"]
    assert obs == 20183
    se = np.hypot(pub["stddev"] / np.sqrt(1000), pub["stddev"] / np.sqrt(500))
    assert abs(r.expected - pub["expected"]) < 4 * se, r.expected
    assert abs(r.stddev - pub["stddev"]) / pub["stddev"] < 0.2
    assert abs(r.fold - pub["fold"]) / pub["fold"] < 0.1
    assert r.pvalue == pytest.approx(1.0 / 500)
    # the row prints through the result objects of gat_b200, which restate the reference's formatting
    row = Engine.AnnotatorResult(track, annotation, counter, obs, samples)
    assert str(row).split("\t")[:3] == [track, annotation, "20183"]


@pytest.mark.parametrize("tag", ["plain", "iso"])
def test_reference_run_equals_package_run_and_reference_distribution(ctx, ref, oracle, tag):
    """one seed, two drivers: the binding (reference-shaped containers, the reference's call sequence) and
    gat_b200.run() produce the SAME sample columns (same library calls underneath), and the expectation agrees with
    the 2000 samples the reference drew with its own sampler (tests/golden/distribution.npz) within 3.5 SE"""
    import gat_b200
    from gat_b200 import engine as Engine
    gat, binding = ref
    z, meta = G.load_npz("distribution")
    m = meta[tag]
    segments = G.collection(z, tag + "/segments", m["segments"])
    annotations = G.collection(z, tag + "/annotations", m["annotations"])
    workspace = G.dictionary(z, tag + "/workspace", m["workspace"])
    names = ["nucleotide-overlap", "segment-overlap"]
    S = 400
    binding.seed(21)
    ref_results = _run(gat, segments, annotations, workspace, names, S)
    Engine.seed(21)
    own = gat_b200.run(segments, annotations, workspace, Engine.SamplerAnnotator(bucket_size=1, nbuckets=100000),
                       [Engine.COUNTER_CLASSES[n]() for n in names], Engine.UnconditionalWorkspace(), num_samples=S)
    own = dict(((r.track, r.annotation, r.counter), r) for r in own)
    assert len(ref_results) == len(own) > 0
    for key, (obs, samples) in ref_results.items():
        o = own[key]
        assert obs == o.observed
        assert np.array_equal(samples, o.samples), key
        st = oracle.enrichment_statistics(obs, samples)
        assert st.pvalue == o.pvalue and st.expected == pytest.approx(o.expected, rel=1e-12)
    # against the reference's own sampler: tests/golden/distribution.npz holds its per-sample counts
    ref_samples = z[tag + "/samples/nucleotide-overlap"]        # [n_samples][n_annotations]
    for (track, annotation, counter), (obs, samples) in ref_results.items():
        if counter != "nucleotide-overlap":
            continue
        col = ref_samples[:, m["annotation_order"].index(annotation)].astype(np.float64)
        se = np.hypot(col.std() / np.sqrt(len(col)), samples.std() / np.sqrt(S))
        assert abs(col.mean() - samples.mean()) <= 3.5 * se + 1e-9, (annotation, col.mean(), samples.mean())
