"""gat-compare: compare the fold changes of two or more GAT runs (mirror of scripts/gat-compare.py).

    python -m gat_b200.compare [options] counts1.tsv [counts2.tsv ...]

The inputs are count tables written with --output-counts-pattern.  With one file every pair of annotations
is compared; with several files the shared (track, annotation) rows of every pair of files.  For a pair the
test statistic is the difference of the two fold changes; its null distribution is the sampled
log(fc1 / fc2) shifted by the observed difference (scripts/gat-compare.py:218-241, :300-323).  The statistics
of every row of every file and of every pair are computed on the GPU in batches (gatb_column_stats,
gatb_compare_stats); q-values and table output are those of gat-run.
"""
import itertools
import optparse
import sys

import numpy as np

from . import engine as Engine
from . import io as IO


def buildParser():
    """options of scripts/gat-compare.py:111-156 plus the -S/-L/-v output options of Experiment.Start"""
    p = optparse.OptionParser(usage=__doc__)
    p.add_option("-o", "--order", dest="output_order", type="choice",
                 choices=("track", "annotation", "fold", "pvalue", "qvalue", "observed"),
                 help="order results in output by fold, track, etc. [default=%default].")
    p.add_option("-p", "--pvalue-method", dest="pvalue_method", type="choice", choices=("empirical", "norm"),
                 help="type of pvalue reported [default=%default].")
    p.add_option("-q", "--qvalue-method", dest="qvalue_method", type="choice",
                 choices=("storey", "BH", "bonferroni", "holm", "hommel", "hochberg", "BY", "none"),
                 help="method to perform multiple testing correction by controlling the fdr [default=%default].")
    p.add_option("--qvalue-lambda", dest="qvalue_lambda", type="float", help="fdr computation: lambda.")
    p.add_option("--qvalue-pi0-method", dest="qvalue_pi0_method", type="choice", choices=("smoother", "bootstrap"),
                 help="fdr computation: method for estimating pi0 [default=%default].")
    p.add_option("--descriptions", dest="input_filename_descriptions", type="string",
                 help="filename mapping annotation terms to descriptions.")
    p.add_option("--pseudo-count", dest="pseudo_count", type="float",
                 help="pseudo count added to the sampled overlap before the fold change [default=%default].")
    p.add_option("--output-plots-pattern", dest="output_plots_pattern", type="string",
                 help="accepted for compatibility; plotting is not part of this path.")
    p.add_option("-S", "--stdout", dest="stdout_file", type="string", default=None, help="output file")
    p.add_option("-L", "--log", dest="log_file", type="string", default=None, help="log file (ignored)")
    p.add_option("-v", "--verbose", dest="loglevel", type="int", default=1, help="log level")
    p.set_defaults(pvalue_method="empirical", qvalue_method="BH", qvalue_lambda=None,
                   qvalue_pi0_method="smoother", pseudo_count=1.0, output_order="observed",
                   output_tables_pattern="%s.tsv.gz")
    return p


def fromCountsBatched(filename):
    """gat.fromCounts (gat/__init__.py:1091-1119) with ONE statistics call for all rows of the file.
    -> (results, matrix [n_samples][n_rows]): the uint32 SampleMatrix of the GPU reader (Engine.readCountsTable), or
    the float64 host array of _fromCountsHost for tables that reader does not take"""
    table = Engine.readCountsTable(filename)
    if table is None:
        return _fromCountsHost(filename)
    rows, matrix = table
    st = Engine.getContext().column_stats(None, [r[2] for r in rows], pseudo_count=1.0,
                                          device_ptr=matrix._tensor.data_ptr(), n_samples=matrix.nsamples,
                                          n_cols=matrix.ncolumns, is_float=0)
    results = [Engine.AnnotatorResult(track, annotation, "na", observed, (matrix, i),
                                      stats=dict((k, float(v[i])) for k, v in st.items()))
               for i, (track, annotation, observed) in enumerate(rows)]
    return results, matrix


def _fromCountsHost(filename):
    """fromCountsBatched parsed on the host, line by line -> (results, matrix [n_samples][n_rows] float64)"""
    rows = []
    with IO.openFile(filename, "r") as infile:
        header = infile.readline()
        if not header == "track\tannotation\tobserved\tcounts\n":
            raise ValueError("%s not a counts file: got %s" % (infile, header))
        for line in infile:
            track, annotation, observed, counts = line[:-1].split("\t")
            rows.append((track, annotation, float(observed),
                         np.array(list(map(float, counts.split(","))), dtype=np.float64)))
    if not rows:
        return [], np.zeros((0, 0))
    if len(set(len(r[3]) for r in rows)) != 1:
        raise ValueError("%s: rows differ in the number of samples" % filename)
    matrix = np.ascontiguousarray(np.stack([r[3] for r in rows], axis=1))
    st = Engine.getContext().column_stats(_as_counts(matrix), [r[2] for r in rows], pseudo_count=1.0)
    results = []
    for i, (track, annotation, observed, samples) in enumerate(rows):
        results.append(Engine.AnnotatorResult(track, annotation, "na", observed, samples,
                                              stats=dict((k, float(v[i])) for k, v in st.items())))
    return results, matrix


def _as_counts(matrix):
    """integer-valued tables go through the exact integer statistics path"""
    if matrix.size and np.all(matrix == np.floor(matrix)) and matrix.min() >= 0 and matrix.max() < 2 ** 32:
        return matrix.astype(np.uint32)
    return matrix


def _nsamples(matrix):
    """samples of a host array or of a SampleMatrix"""
    return matrix.nsamples if isinstance(matrix, Engine.SampleMatrix) else matrix.shape[0]


def comparePairs(pairs, m1, m2, pseudo_count):
    """pairs: [(track, annotation, data1, col1, data2, col2)] -> AnnotatorResult per pair, statistics batched"""
    if not pairs:
        return []
    delta = np.array([p[4].fold - p[2].fold for p in pairs], dtype=np.float64)
    st = Engine.getContext().compare_stats(
        m1, m2, [p[3] for p in pairs], [p[5] for p in pairs], [p[2].observed for p in pairs],
        [p[4].observed for p in pairs], delta, pseudo_count=pseudo_count)
    return [PairResult(track, annotation, 0.0 + delta[i], d1, d2, pseudo_count,
                       dict((k, float(v[i])) for k, v in st.items()))
            for i, (track, annotation, d1, c1, d2, c2) in enumerate(pairs)]


class PairResult(Engine.AnnotatorResult):
    """AnnotatorResult(track, annotation, "na", observed_delta_fold, sampled_delta_fold, pseudo_count=0) whose
    statistics came from the batched GPU call; the derived samples themselves stay on the GPU and are only
    re-derived here if somebody asks for them"""

    def __init__(self, track, annotation, observed, data1, data2, pseudo_count, stats):
        self.track, self.annotation, self.counter = track, annotation, "na"
        self.observed = float(observed)
        self.nsamples = data1.nsamples
        self.format_observed = "%6.4f"
        self.qvalue = 1.0
        self._pair = (data1, data2, pseudo_count)
        for k in ("expected", "stddev", "lower95", "upper95", "fold", "pvalue"):
            setattr(self, k, stats[k])

    @property
    def _source(self):
        d1, d2, pc = self._pair
        with np.errstate(divide="ignore", invalid="ignore"):
            fc1 = d1.observed / (d1.samples + pc) + 0.0001
            fc2 = d2.observed / (d2.samples + pc) + 0.0001
            return np.log(fc1 / fc2) + self.observed


def main(argv=None):
    argv = sys.argv if argv is None else argv
    options, filenames = buildParser().parse_args(argv[1:])
    options.stdout = open(options.stdout_file, "w") if options.stdout_file else sys.stdout
    description_header, descriptions, description_width = IO.readDescriptions(options)

    loaded = []
    for fn in filenames:
        results, matrix = fromCountsBatched(fn)
        if options.pvalue_method != "empirical":
            Engine.updatePValues(results, options.pvalue_method)
        Engine.updateQValues(results, method=options.qvalue_method, vlambda=options.qvalue_lambda,
                             pi0_method=options.qvalue_pi0_method)
        loaded.append((results, matrix))

    results = []
    if len(loaded) == 1:
        annotator_results, matrix = loaded[0]
        if len(set(x.track for x in annotator_results)) != 1:
            raise NotImplementedError("multiple segments of interest")
        idx = range(len(annotator_results))
        pairs = [(annotator_results[i].annotation, annotator_results[j].annotation, annotator_results[i], i,
                  annotator_results[j], j) for i, j in itertools.combinations(idx, 2)]
        results = comparePairs(pairs, matrix, None, options.pseudo_count)
    else:
        for i1, i2 in itertools.combinations(range(len(loaded)), 2):
            (a, ma), (b, mb) = loaded[i1], loaded[i2]
            if _nsamples(ma) != _nsamples(mb):
                raise ValueError("count tables differ in the number of samples")
            aa = dict(((x.track, x.annotation), (x, i)) for i, x in enumerate(a))
            bb = dict(((x.track, x.annotation), (x, i)) for i, x in enumerate(b))
            shared = sorted(set(aa).intersection(bb))
            pairs = [(t, n, aa[(t, n)][0], aa[(t, n)][1], bb[(t, n)][0], bb[(t, n)][1]) for t, n in shared]
            results.extend(comparePairs(pairs, ma, mb, options.pseudo_count))

    if len(results) == 0:
        sys.stderr.write("no results found\n")
        return 0
    IO.outputResults(results, options, Engine.AnnotatorResult.headers, description_header, description_width,
                     descriptions, format_observed="%6.4f")
    if options.stdout_file:
        options.stdout.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
