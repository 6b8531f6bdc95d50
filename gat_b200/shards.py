"""Sharded runs: ranges of the global samples as separate jobs, merged exactly into the results of one run.

    python -m gat_b200.cli <gat-run flags> --random-seed=1 --sample-range=0:50000 --output-shard=part0.npz
    ...
    python -m gat_b200.shards [-o fold] [-q BH] [-p empirical] [--output-tables-pattern=...] [--descriptions=...]
        [-S out.tsv] part*.npz

A shard job (gat_b200.runShard) samples the global sample indices [begin, end) of a run and writes one .npz file
with the exact integer state of every (segment track, counter): the sums of matrixfree.shard_states and the
histogram of every column over its [min, max] in the shard, as sparse CSR.  Every sample is a function of (seed,
track, unit, global sample index), so shards of the same inputs and seed whose ranges tile [0, num_samples), in any
order, merge (mergeShards) into the statistics of run() over all samples, bit for bit; the merge samples nothing.

    python -m gat_b200.shards --combine=OUT part*.npz       # one shard file for the shards' contiguous range
    python -m gat_b200.shards [output flags] --prefix part*.npz

Shards whose ranges form one contiguous [b, e) combine (combineShards) into the shard file a job over [b, e) would
write, so finished shards can be folded together as they arrive.  Shards that tile [0, k) hold exactly the samples of
run(..., num_samples=k): mergeShardPrefix reads the results of the first k samples from the shards that have
finished, up to the first missing range.
"""
import hashlib
import sys

import numpy as np

from . import engine as Engine
from . import matrixfree

FORMAT = "gat_b200 shard"
FORMAT_VERSION = 1

# the size / overlap columns of AnnotatorResultExtended, per result row
SIZES = ("track_nsegments", "track_size", "annotation_nsegments", "annotation_size", "overlap_nsegments",
         "overlap_size", "workspace_size")
STATE = ("rows", "moments", "minmax", "col_ptr", "value", "count")


def inputDigest(sampler, segments, workspace):
    """sha256 over the sampler kind and parameters, the prepared segment lists of every track and the workspace lists
    with their keys (contig or contig.isochore), in iteration order: what the samples are a function of besides the
    seed"""
    h = hashlib.sha256()
    params = (getattr(sampler, "kind", "annotator"), getattr(sampler, "bucket_size", None),
              getattr(sampler, "nbuckets", None), getattr(sampler, "radius", None), getattr(sampler, "extension", None))
    h.update(repr(params).encode())
    for track in segments.tracks:
        h.update(b"\0track\0" + str(track).encode())
        for key, s in segments[track].items():
            h.update(b"\0key\0" + str(key).encode())
            h.update(np.ascontiguousarray(s.asarray(), dtype=np.uint32).tobytes())
    h.update(b"\0workspace\0")
    for key, s in workspace.items():
        h.update(b"\0key\0" + str(key).encode())
        h.update(np.ascontiguousarray(s.asarray(), dtype=np.uint32).tobytes())
    return h.hexdigest()


def writeShard(filename, job, sampled, sizes):
    """the shard file of a shard job (gat_b200._run): metadata, one row per result of run() in run()'s order, and the
    integer state of every (track, counter); sampled[track].planes holds the shard_states"""
    anno_sizes, track_sizes, workspace_size = sizes
    counters = [c.name for c in job.counters]
    tracks = list(sampled.keys())
    atracks = list(job.annotations.tracks)
    rows = dict((k, []) for k in ("counter", "track", "annotation", "observed", "ref_fold") + SIZES)
    for ci in range(len(counters)):
        for track, r in job.observed[ci].items():
            if track not in sampled:
                continue
            for ai, annotation in enumerate(sampled[track].atracks):
                rows["counter"].append(ci)
                rows["track"].append(tracks.index(track))
                rows["annotation"].append(atracks.index(annotation))
                rows["observed"].append(float(r[annotation]))
                rows["ref_fold"].append(job.reference[track][annotation].fold if job.reference else np.nan)
                for k, v in zip(SIZES, (track_sizes[track][0], track_sizes[track][1], anno_sizes[annotation][0],
                                        anno_sizes[annotation][1], track_sizes[track][2][annotation][0],
                                        track_sizes[track][2][annotation][1], workspace_size)):
                    rows[k].append(int(v))
    out = dict(format=np.array(FORMAT), version=np.int64(FORMAT_VERSION), seed=np.uint64(Engine.getSeed()),
               num_samples=np.int64(job.num_samples), sample_range=np.array(job.shard, dtype=np.int64),
               pseudo_count=np.float64(job.pseudo_count), has_reference=np.bool_(bool(job.reference)),
               counters=np.array(counters, dtype=str), tracks=np.array(tracks, dtype=str),
               annotations=np.array(atracks, dtype=str),
               digest=np.array(inputDigest(job.sampler, job.segments, job.workspace)))
    for k in ("counter", "track", "annotation") + SIZES:
        out["row_" + k] = np.array(rows[k], dtype=np.int64)
    out["row_observed"] = np.array(rows["observed"], dtype=np.float64)
    out["row_ref_fold"] = np.array(rows["ref_fold"], dtype=np.float64)
    for ti, track in enumerate(tracks):
        for ci, st in enumerate(sampled[track].planes):
            for k in STATE:
                out["state_%i_%i_%s" % (ti, ci, k)] = np.asarray(st[k])
    _save(filename, out)


def _save(filename, arrays):
    # (np.savez appends .npz to a name without it: write through a file object, so the file is the name given)
    with open(filename, "wb") as f:
        np.savez(f, **arrays)


class Shard(object):
    """one shard file, read and checked for the fields every shard of a run must have"""

    META = ("version", "seed", "num_samples", "sample_range", "pseudo_count", "has_reference", "counters", "tracks",
            "annotations", "digest")

    def __init__(self, filename):
        self.filename = filename
        try:
            with np.load(filename, allow_pickle=False) as z:
                self.arrays = dict((k, z[k]) for k in z.files)
        except Exception as e:
            raise ValueError("%s is not a gat_b200 shard file (%s)" % (filename, e))
        a = self.arrays
        if "format" not in a or str(a["format"]) != FORMAT:
            raise ValueError("%s is not a gat_b200 shard file" % filename)
        if int(a["version"]) != FORMAT_VERSION:
            raise ValueError("%s is a shard of format version %i; this gat_b200 reads version %i"
                             % (filename, int(a["version"]), FORMAT_VERSION))
        self.begin, self.end = (int(x) for x in a["sample_range"])
        self.num_samples = int(a["num_samples"])
        self.counters = [str(x) for x in a["counters"]]
        self.tracks = [str(x) for x in a["tracks"]]
        self.annotations = [str(x) for x in a["annotations"]]

    def state(self, ti, ci):
        return dict((k, self.arrays["state_%i_%i_%s" % (ti, ci, k)]) for k in STATE)


def _same(x, y):
    x, y = np.asarray(x), np.asarray(y)
    return x.shape == y.shape and x.dtype.kind == y.dtype.kind and \
        bool(np.all((x == y) | ((x != x) & (y != y)) if x.dtype.kind == "f" else x == y))


def _readRun(filenames):
    """-> [Shard], checked to be shards of one run (their ranges are not looked at); ValueError naming the files
    otherwise"""
    if not filenames:
        raise ValueError("no shard files given")
    shards = [Shard(f) for f in filenames]
    first = shards[0]
    row_fields = [k for k in first.arrays if k.startswith("row_")]
    for s in shards[1:]:
        for k in Shard.META:
            if k != "sample_range" and not _same(first.arrays[k], s.arrays[k]):
                raise ValueError("%s and %s are not shards of the same run: their %s differ" % (first.filename,
                                                                                                s.filename, k))
        if sorted(k for k in s.arrays if k.startswith("row_")) != sorted(row_fields) or \
                not all(_same(first.arrays[k], s.arrays[k]) for k in row_fields):
            raise ValueError("%s and %s are not shards of the same run: their observed counts, reference folds or "
                             "size columns differ" % (first.filename, s.filename))
    return shards


def _inRange(order):
    """order: shards sorted by range; ValueError for a range that is empty or reaches outside [0, num_samples)"""
    if not 0 <= order[0].begin:
        raise ValueError("%s: sample range starts below 0" % order[0].filename)
    for s in order:
        if s.end <= s.begin:
            raise ValueError("%s: empty sample range [%i, %i)" % (s.filename, s.begin, s.end))
        if s.end > s.num_samples:
            raise ValueError("%s: sample range [%i, %i) ends past num_samples = %i" % (s.filename, s.begin, s.end,
                                                                                       s.num_samples))


def _byRange(shards):
    return sorted(shards, key=lambda s: (s.begin, s.end))


def readShards(filenames):
    """-> [Shard], checked to be shards of one run whose ranges tile [0, num_samples) (in any order); ValueError
    naming the files otherwise"""
    shards = _readRun(filenames)
    first = shards[0]
    order = _byRange(shards)
    if not 0 <= order[0].begin:
        raise ValueError("%s: sample range starts below 0" % order[0].filename)
    at, prev = 0, None
    for s in order:
        if s.end <= s.begin:
            raise ValueError("%s: empty sample range [%i, %i)" % (s.filename, s.begin, s.end))
        if s.begin < at:
            raise ValueError("%s and %s overlap: samples [%i, %i)" % (prev.filename, s.filename, s.begin, at))
        if s.begin > at:
            raise ValueError("samples [%i, %i) are in no shard (a gap%s)"
                             % (at, s.begin, " between %s and %s" % (prev.filename, s.filename) if prev else
                                " before %s" % s.filename))
        at, prev = s.end, s
    if at != first.num_samples:
        raise ValueError("samples [%i, %i) are in no shard (a gap after %s)" % (at, first.num_samples, prev.filename))
    return shards


def mergeShards(filenames):
    """the results of run() over all samples from the files of its shard jobs (runShard) -> [AnnotatorResultExtended]
    in run()'s order.  The samples are not kept: .samples, getSample and getEmpiricalPValue raise RuntimeError, as
    after run(..., keep_samples=False)."""
    return _merge(readShards(filenames), Engine.getContext())


def _contiguous(order):
    """order: shards sorted by range, each range inside [0, num_samples); ValueError naming the files when two
    overlap or when samples between two are in none"""
    at, prev = order[0].begin, None
    for s in order:
        if prev is not None and s.begin < at:
            raise ValueError("%s and %s overlap: samples [%i, %i)" % (prev.filename, s.filename, s.begin,
                                                                      min(at, s.end)))
        if prev is not None and s.begin > at:
            raise ValueError("samples [%i, %i) are in no shard (a gap between %s and %s)"
                             % (at, s.begin, prev.filename, s.filename))
        at, prev = s.end, s
    return order[0].begin, at


def combineShards(filenames, output):
    """the shard files of one run whose ranges are disjoint and together one contiguous range [b, e), in any order ->
    one shard file `output` for [b, e): the state a shard job over [b, e) writes (summed integers, union [min, max],
    the union histogram, exported from the device).  It is an ordinary shard: mergeShards, combineShards and
    mergeShardPrefix take it, so that shards can be merged as they arrive, or as a tree."""
    shards = _readRun(filenames)
    order = _byRange(shards)
    _inRange(order)
    b, e = _contiguous(order)
    first = shards[0]
    a = first.arrays
    out = dict((k, v) for k, v in a.items() if not k.startswith("state_"))
    out["sample_range"] = np.array([b, e], dtype=np.int64)
    ctx = Engine.getContext()
    row_c, row_t = a["row_counter"], a["row_track"]
    for r0, r1 in _blocks(row_c, row_t):
        ci, ti = int(row_c[r0]), int(row_t[r0])
        ref = a["row_ref_fold"][r0:r1] if bool(a["has_reference"]) else None
        st = matrixfree.combine_shard_states(ctx, first.num_samples, a["row_observed"][r0:r1], ref,
                                             [s.state(ti, ci) for s in shards])
        for k in STATE:
            out["state_%i_%i_%s" % (ti, ci, k)] = np.asarray(st[k])
    _save(output, out)


def mergeShardPrefix(filenames):
    """the results of run(..., num_samples=k) from shard files of a run of num_samples >= k samples -> (k,
    [AnnotatorResultExtended] in run()'s order).  k is the end of the longest run of the shards that tiles [0, k)
    from 0: a campaign whose shard jobs have not all finished can be read up to its first missing range.  Shards
    past that gap are not used; their names are written to stderr.  ValueError naming the files when two ranges
    overlap or no shard starts at 0."""
    shards = _readRun(filenames)
    order = _byRange(shards)
    _inRange(order)
    at, prev = 0, None
    for s in order:
        if prev is not None and s.begin < at:
            raise ValueError("%s and %s overlap: samples [%i, %i)" % (prev.filename, s.filename, s.begin,
                                                                      min(at, s.end)))
        at, prev = max(at, s.end), s
    if order[0].begin != 0:
        raise ValueError("samples [0, %i) are in no shard (a gap before %s)" % (order[0].begin, order[0].filename))
    k, used = 0, []
    for s in order:
        if s.begin != k:
            break
        used.append(s)
        k = s.end
    unused = order[len(used):]
    if unused:
        sys.stderr.write("# gat_b200.shards: samples [%i, %i) are in no shard; not used: %s\n"
                         % (k, unused[0].begin, " ".join(s.filename for s in unused)))
    return k, _merge(used, Engine.getContext(), num_samples=k)


def _merge(shards, ctx, budget_bytes=None, num_samples=None):
    """the results of the shards, whose rows together are the run's first num_samples (default: all) samples"""
    first = shards[0].arrays
    S = int(first["num_samples"]) if num_samples is None else int(num_samples)
    pseudo_count = float(first["pseudo_count"])
    counters, tracks, atracks = shards[0].counters, shards[0].tracks, shards[0].annotations
    row_c, row_t, row_a = first["row_counter"], first["row_track"], first["row_annotation"]
    results = []
    for r0, r1 in _blocks(row_c, row_t):
        ci, ti = int(row_c[r0]), int(row_t[r0])
        obs = first["row_observed"][r0:r1]
        ref = first["row_ref_fold"][r0:r1] if bool(first["has_reference"]) else None
        st = matrixfree.merge_shard_states(ctx, S, obs, ref, [s.state(ti, ci) for s in shards], pseudo_count,
                                           budget_bytes)
        matrix = Engine.SamplesNotKept(S, r1 - r0)
        for i, r in enumerate(range(r0, r1)):
            results.append(Engine.AnnotatorResultExtended(
                track=tracks[ti], annotation=atracks[int(row_a[r])], counter=counters[ci], observed=float(obs[i]),
                samples=(matrix, i), track_segments=None, annotation_segments=None, workspace=None,
                pseudo_count=pseudo_count, stats=dict((k, float(v[i])) for k, v in st.items()),
                sizes=dict((k, int(first["row_" + k][r])) for k in SIZES)))
    return results


def _blocks(row_c, row_t):
    """[r0, r1) of the runs of rows of one (counter, track)"""
    edges = [0] + [r for r in range(1, len(row_c)) if (row_c[r], row_t[r]) != (row_c[r - 1], row_t[r - 1])] + \
        [len(row_c)]
    return [(a, b) for a, b in zip(edges[:-1], edges[1:]) if b > a]


def main(argv=None):
    """print the table of the whole run from its shard files, through the output of gat_b200.cli"""
    import optparse
    from . import cli
    from . import io as IO
    argv = sys.argv if argv is None else argv
    parser = optparse.OptionParser(usage=__doc__)
    wanted = ("output_tables_pattern", "output_order", "qvalue_method", "qvalue_lambda", "qvalue_pi0_method",
              "pvalue_method", "input_filename_descriptions")
    for _, flags, kw in cli._OPTIONS:
        if kw["dest"] in wanted:
            kw = dict(kw)
            kw["help"] = kw.get("help", "") + " [default=%default]"
            parser.add_option(*flags, **kw)
    parser.set_defaults(**dict((k, cli._DEFAULTS[k]) for k in wanted))
    parser.add_option("-v", "--verbose", dest="loglevel", type="int", default=1, help="log level")
    parser.add_option("-S", "--stdout", dest="stdout_file", type="string", default=None, help="output file")
    parser.add_option("--combine", dest="combine", type="string", default=None,
                      help="write the shards, whose ranges must form one contiguous range, as one shard file COMBINE "
                      "instead of printing a table")
    parser.add_option("--prefix", dest="prefix", action="store_true", default=False,
                      help="print the table of the run of the first k samples, k the end of the shards' ranges that "
                      "tile [0, k) from 0, instead of requiring them to tile all samples")
    options, filenames = parser.parse_args(argv[1:])
    if not filenames:
        parser.error("no shard files given")
    if options.combine and options.prefix:
        parser.error("--combine and --prefix exclude each other")
    if options.combine:
        combineShards(filenames, options.combine)
        return 0
    if "%s" not in options.output_tables_pattern:
        raise ValueError("output_tables_pattern should contain at least one '%s'")
    options.stdout = open(options.stdout_file, "w") if options.stdout_file else sys.stdout
    description_header, descriptions, description_width = IO.readDescriptions(options)
    if options.prefix:
        k, results = mergeShardPrefix(filenames)
        with np.load(filenames[0], allow_pickle=False) as z:
            n = int(z["num_samples"])
        sys.stderr.write("# gat_b200.shards: samples [0, %i) of %i\n" % (k, n))
    else:
        results = mergeShards(filenames)
    if options.pvalue_method != "empirical":
        Engine.updatePValues(results, options.pvalue_method)
    IO.outputResults(results, options, Engine.AnnotatorResultExtended.headers, description_header, description_width,
                     descriptions)
    if options.stdout_file:
        options.stdout.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
