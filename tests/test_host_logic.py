"""CPU tests of the host-side mirror: SegmentList / containers (input preparation), multiple-testing
correction, flag parser.  Pinned against golden vectors of the reference (tests/golden/)."""
import io
import os

import numpy as np
import pytest

from tests import golden_util as G
from gat_b200.segmentlist import SegmentList
from gat_b200 import engine as Engine
from gat_b200 import stats as Stats


def SL(x, normalize=True):
    return SegmentList(iter=[tuple(t) for t in x], normalize=normalize)


def test_segmentlist_matches_reference():
    for c in G.load_json("segmentlist"):
        na, nb = SL(c["a"]), SL(c["b"])
        assert na.asList() == [tuple(x) for x in c["normalize_a"]]
        for d in (0, 1, 5):
            m = SL(c["a"], normalize=False)
            m.merge(d)
            assert m.asList() == [tuple(x) for x in c["merge_%i" % d]]
        f = na.clone()
        f.filter(nb)
        assert f.asList() == [tuple(x) for x in c["filter"]]
        i = na.clone()
        i.intersect(nb)
        assert i.asList() == [tuple(x) for x in c["intersect"]]
        assert na.sum() == c["sum_a"]
        assert na.overlapWithSegments(nb) == c["overlap"]
        assert na.intersectionWithSegments(nb) == c["isect_base"]
        assert na.intersectionWithSegments(nb, mode="midpoint") == c["isect_mid"]
        for bucket in (0, 1, 4):
            key = "lengthdist_%i" % bucket
            if key not in c:
                continue
            if "error" in c[key]:
                with pytest.raises(ValueError):
                    na.getLengthDistribution(bucket, 1000)
                continue
            h, bs = na.getLengthDistribution(bucket, 1000)
            assert bs == c[key]["bucket_size"]
            assert [[int(k), int(h[k])] for k in np.flatnonzero(h)] == c[key]["nonzero"]


def test_segmentlist_reference_unit_tests():
    """test/test_SegmentList.py: normalize variants (:27-142), negatives raise OverflowError (:332-366)"""
    assert SL([(0, 10), (10, 20)]).asList() == [(0, 10), (10, 20)]
    assert SL([(0, 10), (9, 20)]).asList() == [(0, 20)]
    s = SegmentList()
    assert s.isNormalized and s.isEmpty and len(s) == 0
    s.add(5, 10)
    assert not s.isNormalized
    s.normalize()
    assert s.isNormalized and s.sum() == 5
    with pytest.raises(OverflowError):
        SegmentList(iter=[(-1, 5)])
    with pytest.raises(ValueError):
        SL([(0, 10), (5, 15)], normalize=False).check()
    e = SL([(0, 10)])
    e.extend(SL([(20, 30)]))
    assert not e.isNormalized and len(e) == 2


def test_isochore_round_trip():
    """toIsochores / fromIsochores (test/test_gat.py:55-114; gat/Engine.pyx:2837-2876)"""
    d = Engine.IntervalDictionary()
    d.add("chr1", SL([(0, 100), (200, 300), (290, 310)]))
    iso = Engine.IntervalCollection("isochores")
    iso.add("lo", "chr1", SL([(0, 150)]))
    iso.add("hi", "chr1", SL([(150, 400)]))
    t = d.clone()
    t.toIsochores(iso, truncate=True)
    assert sorted(t.keys()) == ["chr1.hi", "chr1.lo"]
    assert t["chr1.lo"].asList() == [(0, 100)] and t["chr1.hi"].asList() == [(200, 310)]
    t.fromIsochores()
    assert list(t.keys()) == ["chr1"] and t["chr1"].asList() == [(0, 100), (200, 310)]
    # without truncation a segment spanning two isochores is present in both (quirk C-7) ...
    d2 = Engine.IntervalDictionary()
    d2.add("chr1", SL([(100, 200)]))
    d2.toIsochores(iso, truncate=False)
    assert d2["chr1.lo"].asList() == [(100, 200)] and d2["chr1.hi"].asList() == [(100, 200)]
    # ... and merge(0) joins adjacent pieces on the way back
    d3 = Engine.IntervalDictionary()
    d3.add("chr1", SL([(100, 200)]))
    d3.toIsochores(iso, truncate=True)
    d3.fromIsochores()
    assert d3["chr1"].asList() == [(100, 200)]
    # a key with a second "." cannot be split into (contig, isochore): ValueError, as in the reference
    # (gat/Engine.pyx:2864-2865; SURVEY quirk C-13)
    d4 = Engine.IntervalDictionary()
    d4.add("chr1.random.lo", SL([(0, 10)]))
    with pytest.raises(ValueError):
        d4.fromIsochores()


def test_truncating_isochore_split_equals_per_track_intersections():
    """toIsochores(truncate=True) splits a contig's list over all isochore tracks in one pass when the tracks do
    not overlap each other; the lists must be those of the reference's loop `clone(); intersect(iso[contig])`
    per track (gat/Engine.pyx:2845-2852) -- random partitions, gaps, overlapping tracks (per-track path), empty
    lists, and several tracks of a collection sharing the cached pieces"""
    from tests import helpers

    def sl(a):
        x = SegmentList(array=a)
        x._normalized = True
        return x
    rng = np.random.default_rng(9)
    for it in range(150):
        span = int(rng.choice([3000, 100000]))
        niso = int(rng.integers(1, 5))
        iso = Engine.IntervalCollection("iso")
        if it % 5 == 0:                               # independent random lists: tracks may overlap each other
            for i in range(niso):
                iso.add("g%i" % i, "c", sl(helpers.random_list(rng, span, int(rng.integers(0, 8)), span // 6)))
        else:                                         # tiles dealt to the tracks, some left out (gaps)
            bounds = np.arange(0, span + 1, span // 20)
            lab = rng.integers(0, niso + 1, len(bounds) - 1)
            for i in range(niso):
                m = lab == i
                iso.add("g%i" % i, "c", sl(helpers.normalize(np.stack([bounds[:-1][m], bounds[1:][m]], axis=1))))
        coll = Engine.IntervalCollection("x")
        lists = {}
        for t in range(3):
            lists[t] = helpers.random_list(rng, span, int(rng.integers(0, 60)), int(rng.choice([20, 400, 5000])))
            coll.add("t%i" % t, "c", sl(lists[t].copy()))
        coll.toIsochores(iso, truncate=True)
        for t in range(3):
            got = coll["t%i" % t]
            assert sorted(got.keys()) == sorted("c.%s" % k for k in iso.keys())
            for k, vv in iso.items():
                want = sl(lists[t].copy())
                want.intersect(vv["c"])
                assert got["c.%s" % k].asList() == want.asList(), (it, t, k)
                assert got["c.%s" % k].isNormalized


def test_collection_collapse_merge_restrict():
    c = Engine.IntervalCollection("ws")
    c.add("a", "chr1", SL([(0, 100)]))
    c.add("a", "chr2", SL([(0, 50)]))
    c.add("b", "chr1", SL([(50, 150)]))
    c.collapse()
    assert c["collapsed"]["chr1"].asList() == [(50, 100)] and "chr2" not in c["collapsed"]
    c.restrict("collapsed")
    assert list(c.tracks) == ["collapsed"]
    m = Engine.IntervalCollection("s")
    m.add("x", "chr1", SL([(0, 10)]))
    m.add("y", "chr1", SL([(5, 20)]))
    m.merge()
    assert len(m["merged"]["chr1"]) == 2 and m.countsPerTrack()["merged"] == 2


def test_adjust_pvalues_match_reference():
    for c in G.load_json("qvalues"):
        for method, want in c["adjusted"].items():
            assert np.array_equal(Stats.adjustPValues(c["pvalues"], method=method), np.array(want)), method


def test_storey_qvalues_match_reference():
    n = 0
    for c in G.load_json("qvalues"):
        if "storey_lambda05" in c:
            r = Stats.computeQValues(c["pvalues"], vlambda=0.5)
            assert r.pi0 == pytest.approx(c["storey_lambda05"]["pi0"], rel=1e-14)
            assert np.allclose(r.qvalues, c["storey_lambda05"]["qvalues"], rtol=1e-13, atol=0)
            n += 1
        if "storey_smoother" in c and "qvalues" in c["storey_smoother"]:
            r = Stats.computeQValues(c["pvalues"], vlambda=np.arange(0, 0.95, 0.05), pi0_method="smoother")
            assert r.pi0 == pytest.approx(c["storey_smoother"]["pi0"], rel=1e-12)
            assert np.allclose(r.qvalues, c["storey_smoother"]["qvalues"], rtol=1e-12, atol=0)
            n += 1
    assert n >= 4
    with pytest.raises(ValueError):
        Stats.computeQValues([0.5, 1.5])
    assert Engine.getQValues([0.01, 0.5, 0.9], method="BH")[0] == pytest.approx(0.03)


def test_parser_flags_and_defaults():
    """the flags north_star names and the reference's defaults (gat/__init__.py:385-427)"""
    import gat_b200
    p = gat_b200.buildParser()
    o, _ = p.parse_args(["--segments=s.bed", "--annotations=a.bed", "--workspace=w.bed", "--isochore-file=i.bed",
                         "--counter=segment-overlap", "--num-samples=77", "--sampler=annotator"])
    assert o.segment_files == ["s.bed"] and o.annotation_files == ["a.bed"] and o.workspace_files == ["w.bed"]
    assert o.isochore_files == ["i.bed"] and o.counters == ["segment-overlap"] and o.num_samples == 77
    d, _ = gat_b200.buildParser().parse_args([])      # fresh parser: optparse shares list defaults
    assert (d.num_samples, d.bucket_size, d.nbuckets, d.pseudo_count) == (1000, 0, 100000, 1.0)
    assert d.ignore_segment_tracks is True and d.qvalue_method == "BH" and d.sampler == "annotator"
    assert d.output_order == "fold" and d.pvalue_method == "empirical" and d.counters == []


def test_parser_equals_reference_option_for_option():
    """buildParser() offers every option of the reference's gat.buildParser() with the same flags, action, type,
    choices and default (tests/golden/parser_options.json), and none of its own"""
    import gat_b200
    ref = G.load_json("parser_options")
    p = gat_b200.buildParser()
    mine = {}
    for o in p._get_all_options():
        if o.dest:
            mine[o.dest] = dict(flags=sorted(o._long_opts + o._short_opts), action=o.action, type=o.type,
                                default=p.defaults.get(o.dest), choices=list(o.choices) if o.choices else None)
    assert sorted(mine) == sorted(ref)
    for dest, want in ref.items():
        got = mine[dest]
        for k in ("flags", "action", "type", "choices"):
            assert got[k] == want[k], (dest, k, got[k], want[k])
        # (an absent list default reads as None in the reference and as [] here: both are "no files")
        assert got["default"] == want["default"] or (not got["default"] and not want["default"]), dest


def test_bed_reader_tracks(tmp_path):
    from gat_b200 import io as IO
    f = tmp_path / "x.bed"
    f.write_text("track name=t1\nchr1\t10\t20\nchr1\t15\t30\ntrack name=\"t2\"\nchr2\t0\t5\n")
    r = IO.readFromBed([str(f)])
    assert sorted(r.keys()) == ["t1", "t2"] and r["t1"]["chr1"].asList() == [(10, 20), (15, 30)]
    g = tmp_path / "y.bed"
    g.write_text("chr1\t1\t2\tnameA\nchr1\t3\t4\n")
    r = IO.readFromBed([str(g)])
    assert sorted(r.keys()) == ["nameA", "y.bed"]
    with pytest.raises(ValueError):          # like the reference: one track may not span files ...
        IO.readFromBed([str(f), str(g)], ignore_tracks=True)
    r = IO.readFromBed([str(f), str(g)], ignore_tracks=True, allow_multiple=True)   # ... unless allowed
    assert list(r.keys()) == ["merged"] and r["merged"]["chr1"].counts() == 4


def test_input_preparation_matches_reference_io(tmp_path, monkeypatch):
    """our buildSegments + applyIsochores on the reference's test data == the arrays the reference's own
    IO produced (stored in tests/golden/observed_testdata.npz).  The BED files are written from those arrays
    (segment and annotation tracks in the name column, gzip-compressed like the reference's test/data): reading
    and preparing what the reference prepared must give it back unchanged.  Host preparation (GATB_HOST_PREP=1)."""
    import gzip
    import gat_b200
    from gat_b200 import io as IO
    monkeypatch.setenv("GATB_HOST_PREP", "1")
    z, meta = G.load_npz("observed_testdata")
    d = str(tmp_path)
    for fn, name, keys in (("segments_single.bed.gz", "segments", meta["segments"]),
                           ("annotations.bed.gz", "annotations", meta["annotations"]),
                           ("workspace.bed.gz", "workspace", [(None, k) for k in meta["workspace"]])):
        with gzip.open(os.path.join(d, fn), "wt") as f:
            for track, key in keys:
                arr = z["%s/%s" % (name, key)] if track is None else z["%s/%s/%s" % (name, track, key)]
                for start, end in G.undelta(arr):
                    f.write("%s\t%i\t%i%s\n" % (key, start, end, "" if track is None else "\t" + track))
    options, _ = gat_b200.buildParser().parse_args([
        "--segments=%s/segments_single.bed.gz" % d, "--annotations=%s/annotations.bed.gz" % d,
        "--workspace=%s/workspace.bed.gz" % d, "--with-segment-tracks"])
    segments, annotations, workspaces, isochores = IO.buildSegments(options)
    workspace = IO.applyIsochores(segments, annotations, workspaces, options, isochores)
    assert sorted(workspace.keys()) == sorted(meta["workspace"])
    for key in meta["workspace"]:
        assert np.array_equal(workspace[key].asarray(), G.undelta(z["workspace/%s" % key]))
    for name, coll in (("segments", segments), ("annotations", annotations)):
        # (the fixture was dumped after computeCounts, whose defaultdict look-ups leave empty lists behind
        # for every workspace key: compare the non-empty lists)
        ref_keys = sorted([t, k] for t, k in meta[name] if len(z["%s/%s/%s" % (name, t, k)]))
        assert sorted([t, k] for t, vv in coll.items() for k in vv.keys() if len(vv[k])) == ref_keys
        for track, key in ref_keys:
            assert np.array_equal(coll[track][key].asarray(), G.undelta(z["%s/%s/%s" % (name, track, key)])), (track, key)


def test_isochore_preparation_matches_reference_io(tmp_path, monkeypatch):
    """buildSegments + applyIsochores WITH an isochore file (toIsochores of workspace, annotations and segments,
    gat/IO.py:188-293) give the lists the reference's own IO gave for the same BED files -- default (segments
    filtered per isochore) and --truncate-segments-to-workspace (tests/golden/prep_isochores.json).  Host
    preparation (GATB_HOST_PREP=1) here; tests/test_gpu_prep.py runs the device preparation against the same
    fixture."""
    import gat_b200
    from gat_b200 import io as IO
    monkeypatch.setenv("GATB_HOST_PREP", "1")
    data = G.load_json("prep_isochores")
    argv = []
    for name, flag in (("segments", "--segments"), ("annotations", "--annotations"), ("workspace", "--workspace"),
                       ("iso", "--isochore-file")):
        path = tmp_path / (name + ".bed")
        path.write_text(data["files"][name + ".bed"])
        argv.append("%s=%s" % (flag, path))
    assert len(data["cases"]) == 2
    for case in data["cases"]:
        options, _ = gat_b200.buildParser().parse_args(argv + case["extra"])
        segments, annotations, workspaces, isochores = IO.buildSegments(options)
        workspace = IO.applyIsochores(segments, annotations, workspaces, options, isochores,
                                      truncate_segments_to_workspace=options.truncate_segments_to_workspace)
        assert sorted(workspace.keys()) == sorted(case["workspace"].keys())
        for k, want in case["workspace"].items():
            assert workspace[k].asList() == [tuple(x) for x in want], k
        n = 0
        for name, coll in (("segments", segments), ("annotations", annotations)):
            assert sorted(coll.tracks) == sorted(case[name].keys())
            for track, lists in case[name].items():
                for k, want in lists.items():
                    got = coll[track][k].asList() if k in coll[track] else []
                    assert got == [tuple(x) for x in want], (name, track, k)
                    n += 1
        assert n > 40


def test_result_row_formatting_matches_reference():
    """AnnotatorResult.__str__ (gat/Engine.pyx:1802-1852): built from the reference's own statistics, every
    row prints exactly as the reference printed it (tests/golden/stats.json: integer and float observed values,
    zero expectations, folds <= 0 -> "-inf")"""
    cases = G.load_json("stats")
    n = 0
    for c in cases:
        if c["ref_fold"] is not None:
            continue
        stats = dict((k, c[k]) for k in ("expected", "stddev", "fold", "pvalue", "lower95", "upper95"))
        r = Engine.AnnotatorResult("t", "a", "na", c["observed"], np.array(c["samples"], dtype=np.float64), stats=stats)
        want = c["row"].split("\t")
        got = str(r).split("\t")
        # CI columns of the fixture were parsed back from the printed row (4 decimals): compare the others exactly
        assert got[:4] == want[:4] and got[6:] == want[6:], (got, want)
        assert got[4:6] == want[4:6]
        n += 1
    assert n >= 30


@pytest.mark.parametrize("tag", ["plain", "iso"])
def test_extended_result_rows_match_reference(tag):
    """AnnotatorResultExtended (gat/Engine.pyx:1854-1974): the size / overlap / density / percent columns computed on
    the host from the prepared lists, and the whole printed row, equal the rows of the reference's own small runs
    (tests/golden/run_small.npz; statistics and q-value are taken from the fixture, so no GPU is involved)"""
    z, meta = G.load_npz("run_small")
    m = meta[tag]
    segments = G.collection(z, tag + "/segments", m["segments"])
    annotations = G.collection(z, tag + "/annotations", m["annotations"])
    workspace = G.dictionary(z, tag + "/workspace", m["workspace"])
    n = 0
    for counter, per_annotation in m["results"].items():
        for annotation, ref in per_annotation.items():
            want = ref["row"].split("\t")
            stats = dict(expected=ref["expected"], stddev=ref["stddev"], fold=ref["fold"], pvalue=ref["pvalue"],
                         lower95=float(want[4]), upper95=float(want[5]))
            r = Engine.AnnotatorResultExtended(want[0], annotation, counter, ref["observed"],
                                               np.array(ref["samples"]), segments[want[0]], annotations[annotation],
                                               workspace, stats=stats)
            r.qvalue = float(want[10])
            if counter == "nucleotide-density":
                r.format_observed = "%6.4e" if "e" in want[2] else r.format_observed
            got = str(r).split("\t")
            assert len(got) == len(Engine.AnnotatorResultExtended.headers) == len(want)
            assert got[11:] == want[11:], (counter, annotation, got[11:], want[11:])
            assert got[:2] == want[:2] and got[3:11] == want[3:11], (counter, annotation)
            n += 1
    assert n >= 12


def test_output_tables_match_reference(tmp_path):
    """IO.outputResults (gat/IO.py:457-538): q-values over all results of the run, one table per counter, rows in
    --output-order, optional annotation descriptions -- the text equals what the reference wrote for its own
    results (tests/golden/output_tables.json: six orders x {BH, storey, BH with descriptions})"""
    from gat_b200 import io as IO
    data = G.load_json("output_tables")
    sizes_keys = ("track_nsegments", "track_size", "annotation_nsegments", "annotation_size", "overlap_nsegments",
                  "overlap_size")
    assert data["headers"] == Engine.AnnotatorResultExtended.headers

    def build():
        res = []
        for r in data["results"]:
            tail = r["tail"]
            sizes = dict(zip(sizes_keys, [int(tail[0]), int(tail[1]), int(tail[3]), int(tail[4]), int(tail[6]), int(tail[7])]))
            sizes["workspace_size"] = data["workspace_size"]
            stats = dict((k, r[k]) for k in ("expected", "stddev", "fold", "pvalue", "lower95", "upper95"))
            res.append(Engine.AnnotatorResultExtended(r["track"], r["annotation"], r["counter"], r["observed"],
                                                      np.zeros(1), None, None, None, stats=stats, sizes=sizes))
        return res

    for case in data["cases"]:
        class O(object):
            pass
        O.qvalue_method, O.qvalue_lambda, O.qvalue_pi0_method = case["method"], None, "smoother"
        O.output_order = case["order"]
        O.output_tables_pattern = str(tmp_path / "t_%s.tsv")
        desc = data["descriptions"] if case["with_desc"] else {}
        IO.outputResults(build(), O, Engine.AnnotatorResultExtended.headers,
                         ["description", "extra"] if case["with_desc"] else [], 2 if case["with_desc"] else 0, desc)
        for counter, want in case["tables"].items():
            got = open(str(tmp_path / ("t_%s.tsv" % counter))).read()
            assert got == want, (case["order"], case["method"], case["with_desc"], counter)


def test_bed_fast_reader_equals_line_reader(tmp_path, monkeypatch):
    """the Arrow fast path of IO.readFromBed and the line-by-line reader give the same tracks, the same key
    order and the same intervals; files it cannot take (track lines, comments, ragged rows) fall back"""
    import gzip
    from gat_b200 import io as IO
    rng = np.random.default_rng(12)
    contigs = ["chr2", "chr1", "chrX", "chr10"]
    lines = []
    for i in range(5000):
        s = int(rng.integers(0, 10 ** 8))
        lines.append("%s\t%i\t%i\t%s\n" % (contigs[int(rng.integers(0, 4))], s, s + int(rng.integers(1, 5000)),
                                           ["tB", "tA", "", "tC"][int(rng.integers(0, 4))]))
    plain = str(tmp_path / "plain.bed")
    open(plain, "w").write("".join(lines))
    three = str(tmp_path / "three.bed")
    open(three, "w").write("".join("\t".join(l.split("\t")[:3]) + "\n" for l in lines))
    gz = str(tmp_path / "z.bed.gz")
    with gzip.open(gz, "wt") as f:
        f.write("".join(lines))
    tracked = str(tmp_path / "tracked.bed")
    open(tracked, "w").write("chr1\t5\t9\n# comment\ntrack name=\"q r\"\n" + "".join(lines[:50]) + "track name=z\nchr1\t1\t2\n")

    def both(files, **kw):
        fast = IO.readFromBed(files, **kw)
        with monkeypatch.context() as m:
            m.setattr(IO, "_readBedColumns", lambda fn: None)
            slow = IO.readFromBed(files, **kw)
        assert list(fast.keys()) == list(slow.keys())
        for t in slow:
            assert list(fast[t].keys()) == list(slow[t].keys()), t
            for c in slow[t].keys():
                assert np.array_equal(fast[t][c].asarray(), slow[t][c].asarray()), (t, c)
        return fast

    assert IO._readBedColumns(plain) is not None and IO._readBedColumns(gz) is not None
    assert IO._readBedColumns(tracked) is None
    r = both([plain])
    assert set(r.keys()) == {"tA", "tB", "tC", "plain.bed"}
    assert list(both([three]).keys()) == ["three.bed"]
    assert list(both([gz], ignore_tracks=True).keys()) == ["merged"]
    r = both([tracked])
    assert set(r.keys()) == {"tracked.bed", "q r", "z"}
    both([plain, three, tracked], allow_multiple=True)
    with pytest.raises(ValueError):
        IO.readFromBed([plain, gz])                                # same tracks in two files
