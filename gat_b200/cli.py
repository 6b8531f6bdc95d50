"""Command line of the accelerated path: same flags and defaults as the reference's gat-run.py
(`gat.buildParser`, gat/__init__.py:54-429; `main`, scripts/gat-run.py:223-314).

    python -m gat_b200.cli --segments=s.bed --annotations=a.bed --workspace=w.bed \
        [--isochore-file=i.bed] [--counter=nucleotide-overlap] [--num-samples=1000] [--sampler=annotator]

Multi-GPU: launch with `python -m torch.distributed.run --nproc-per-node N -m gat_b200.cli ...`.

A run in several jobs: `--random-seed=S --sample-range=BEGIN:END --output-shard=FILE` samples only the global samples
[BEGIN, END) of the run and writes their exact state to FILE instead of a table; `python -m gat_b200.shards FILE...`
merges the shards of ranges that tile [0, --num-samples) into the run's table (gat_b200/shards.py).
"""
import optparse
import random
import sys
import time

import numpy as np

COUNTER_CHOICES = ("nucleotide-overlap", "nucleotide-density", "segment-overlap", "segment-midoverlap",
                   "annotation-overlap", "annotation-midoverlap")
SAMPLER_CHOICES = ("annotator", "segments", "shift", "local-permutation", "global-permutation", "uniform",
                   "brute-force")

# (group, flags, kwargs) -- one row per option of the reference parser
_OPTIONS = [
    ("Input options", ("-a", "--annotation-bed-file", "--annotations", "--annotation-file"),
     dict(dest="annotation_files", type="string", action="append", help="filename with annotations")),
    ("Input options", ("-s", "--segment-bed-file", "--segments", "--segment-file"),
     dict(dest="segment_files", type="string", action="append", help="filename with segments")),
    ("Input options", ("-w", "--workspace-bed-file", "--workspace", "--workspace-file"),
     dict(dest="workspace_files", type="string", action="append", help="filename with workspace segments")),
    ("Input options", ("-i", "--isochore-bed-file", "--isochores", "--isochore-file"),
     dict(dest="isochore_files", type="string", action="append", help="filename with isochore segments")),
    ("Input options", ("-l", "--sample-file"),
     dict(dest="sample_files", type="string", action="append", help="start from sample files (not accelerated)")),
    ("Input options", ("--input-counts-file",),
     dict(dest="input_filename_counts", type="string", help="start processing from a counts table")),
    ("Input options", ("--input-results-file",),
     dict(dest="input_filename_results", type="string", help="start processing from a results table")),
    ("Input options", ("--ignore-segment-tracks",),
     dict(dest="ignore_segment_tracks", action="store_true", help="all segments belong to one track 'merged'")),
    ("Input options", ("--with-segment-tracks",),
     dict(dest="ignore_segment_tracks", action="store_false", help="the segments file is arranged in tracks")),
    ("Input options", ("--enable-split-tracks",),
     dict(dest="enable_split_tracks", action="store_true", help="permit one track in several files")),
    ("Input options", ("--overlapping-annotations",),
     dict(dest="overlapping_annotations", action="store_true", help="annotations overlap (not accelerated)")),
    ("Input options", ("--annotations-label",),
     dict(dest="annotations_label", type="string", help="ignore annotation tracks, use this label")),
    ("Input options", ("--annotations-to-points",),
     dict(dest="annotations_to_points", type="choice", choices=("midpoint", "start", "end"),
          help="convert annotations to positions (not accelerated)")),
    ("Output options", ("-o", "--order"),
     dict(dest="output_order", type="choice", choices=("track", "annotation", "fold", "pvalue", "qvalue"),
          help="order of the results table")),
    ("Output options", ("--output-tables-pattern",),
     dict(dest="output_tables_pattern", type="string", help="pattern for result tables with several counters")),
    ("Output options", ("--output-counts-pattern",),
     dict(dest="output_counts_pattern", type="string", help="pattern for the sampled-counts tables")),
    ("Output options", ("--output-plots-pattern",),
     dict(dest="output_plots_pattern", type="string", help="pattern for plots (unused)")),
    ("Output options", ("--output-samples-pattern",),
     dict(dest="output_samples_pattern", type="string", help="pattern for BED files with the samples")),
    ("Output options", ("--output-stats",),
     dict(dest="output_stats", type="choice", action="append",
          choices=("all", "annotations", "segments", "workspaces", "isochores", "overlap", "sample",
                   "segment_metrics", "sample_metrics"), help="summary statistics to output (unused)")),
    ("Output options", ("--output-bed",),
     dict(dest="output_bed", type="choice", action="append",
          choices=("all", "annotations", "segments", "workspaces", "isochores", "overlap"),
          help="bed files to output (unused)")),
    ("Output options", ("--descriptions",),
     dict(dest="input_filename_descriptions", type="string", help="table mapping annotations to descriptions")),
    ("Sampling algorithm options", ("-c", "--counter"),
     dict(dest="counters", type="choice", action="append", choices=COUNTER_CHOICES,
          help="quantity to use for estimating enrichment")),
    ("Sampling algorithm options", ("-m", "--sampler"),
     dict(dest="sampler", type="choice", choices=SAMPLER_CHOICES, help="sampling method (accelerated: annotator)")),
    ("Sampling algorithm options", ("-n", "--num-samples"),
     dict(dest="num_samples", type="int", help="number of samples to compute")),
    ("Sampling algorithm options", ("--shift-extension",), dict(dest="shift_extension", type="float", help="--sampler=shift: size of the window a segment is shifted in, in bases (0 = use --shift-expansion)")),
    ("Sampling algorithm options", ("--shift-expansion",), dict(dest="shift_expansion", type="float", help="--sampler=shift: window as a multiple of the segment length")),
    ("Sampling algorithm options", ("--bucket-size",),
     dict(dest="bucket_size", type="int", help="bin size of the segment length histogram, 0 = automatic")),
    ("Sampling algorithm options", ("--nbuckets",),
     dict(dest="nbuckets", type="int", help="number of bins of the segment length histogram")),
    ("Statistics options", ("-p", "--pvalue-method"),
     dict(dest="pvalue_method", type="choice", choices=("empirical", "norm"), help="type of p-value")),
    ("Statistics options", ("-q", "--qvalue-method"),
     dict(dest="qvalue_method", type="choice",
          choices=("storey", "BH", "bonferroni", "holm", "hommel", "hochberg", "BY", "none"),
          help="multiple testing correction")),
    ("Statistics options", ("--qvalue-lambda",), dict(dest="qvalue_lambda", type="float", help="storey: lambda")),
    ("Statistics options", ("--qvalue-pi0-method",),
     dict(dest="qvalue_pi0_method", type="choice", choices=("smoother", "bootstrap"), help="storey: pi0 method")),
    ("Statistics options", ("--pseudo-count",),
     dict(dest="pseudo_count", type="float", help="pseudo count added to observed and expected")),
    ("Statistics options", ("--null",), dict(dest="null", type="string", help="gat results to test against")),
    ("Processing options", ("-e", "--cache"), dict(dest="cache", type="string", help="unused (dead in the reference)")),
    ("Processing options", ("-t", "--num-threads"),
     dict(dest="num_threads", type="int", help="unused: sampling runs on the GPU")),
    ("Processing options", ("--random-seed",), dict(dest="random_seed", type="int", help="random seed")),
    ("Workspace manipulation (experimental)", ("--conditional",),
     dict(dest="conditional", type="choice",
          choices=("unconditional", "annotation-centered", "segment-centered", "cooccurance"),
          help="conditional workspace (accelerated: unconditional)")),
    ("Workspace manipulation (experimental)", ("--conditional-extension",),
     dict(dest="conditional_extension", type="int", help="unused")),
    ("Workspace manipulation (experimental)", ("--conditional-expansion",),
     dict(dest="conditional_expansion", type="float", help="unused")),
    ("Workspace manipulation (experimental)", ("--restrict-workspace",),
     dict(dest="restrict_workspace", action="store_true", help="keep workspace parts with segments and annotations")),
    ("Workspace manipulation (experimental)", ("--truncate-workspace-to-annotations",),
     dict(dest="truncate_workspace_to_annotations", action="store_true", help="truncate workspace with annotations")),
    ("Workspace manipulation (experimental)", ("--truncate-segments-to-workspace",),
     dict(dest="truncate_segments_to_workspace", action="store_true", help="truncate segments to workspace")),
]

_DEFAULTS = dict(
    annotation_files=[], annotations_label=None, annotations_to_points=None, bucket_size=0, cache=None,
    conditional="unconditional", conditional_expansion=None, conditional_extension=None, counters=[],
    enable_split_tracks=False, ignore_segment_tracks=True, input_filename_counts=None,
    input_filename_descriptions=None, input_filename_results=None, isochore_files=[], nbuckets=100000,
    null="default", num_samples=1000, num_threads=0, output_bed=[], output_counts_pattern=None,
    output_order="fold", output_plots_pattern=None, output_samples_pattern=None, output_stats=[],
    output_tables_pattern="%s.tsv.gz", overlapping_annotations=False, pseudo_count=1.0,
    pvalue_method="empirical", qvalue_lambda=None, qvalue_method="BH", qvalue_pi0_method="smoother",
    random_seed=None, restrict_workspace=False, sample_files=[], sampler="annotator", segment_files=[],
    shift_expansion=2.0, shift_extension=0, truncate_segments_to_workspace=False,
    truncate_workspace_to_annotations=False, workspace_files=[])


def buildParser(usage=None):
    """the gat command line parser: flags, destinations and defaults of gat.buildParser"""
    parser = optparse.OptionParser(version="%prog (gat_b200)", usage=usage)
    groups = {}
    for group, flags, kw in _OPTIONS:
        if group not in groups:
            groups[group] = optparse.OptionGroup(parser, group)
            parser.add_option_group(groups[group])
        kw = dict(kw)
        kw["help"] = kw.get("help", "") + " [default=%default]"
        groups[group].add_option(*flags, **kw)
    parser.set_defaults(**dict((k, (list(v) if isinstance(v, list) else v)) for k, v in _DEFAULTS.items()))
    return parser


def fromSegments(options, log=None, shard=None):
    """load, prepare and run (scripts/gat-run.py:77-220); shard = ((begin, end), filename): write the shard of that
    sample range instead (gat_b200.runShard) -> None"""
    import gat_b200
    from . import io as IO
    from . import engine as Engine

    t0 = time.time()
    segments, annotations, workspaces, isochores = IO.buildSegments(options)
    workspace = IO.applyIsochores(
        segments, annotations, workspaces, options, isochores,
        truncate_segments_to_workspace=options.truncate_segments_to_workspace,
        truncate_workspace_to_annotations=options.truncate_workspace_to_annotations,
        restrict_workspace=options.restrict_workspace)
    if log:
        log("intervals loaded in %.1f seconds" % (time.time() - t0))
    if options.sampler == "annotator":
        sampler = Engine.SamplerAnnotator(bucket_size=options.bucket_size, nbuckets=options.nbuckets)
    elif options.sampler == "segments":
        sampler = Engine.SamplerSegments()
    elif options.sampler == "shift":            # scripts/gat-run.py:129-132
        sampler = Engine.SamplerShift(radius=options.shift_expansion, extension=options.shift_extension)
    else:
        raise NotImplementedError("--sampler=%s is not accelerated by gat_b200 (annotator, segments, shift)" % options.sampler)
    counters = [Engine.COUNTER_CLASSES[c]() for c in options.counters]
    if options.conditional != "unconditional":
        raise NotImplementedError("--conditional=%s is not accelerated by gat_b200" % options.conditional)
    t0 = time.time()
    if log:
        log("sampling started")
    kwargs = dict(num_samples=options.num_samples, output_counts_pattern=options.output_counts_pattern,
                  output_samples_pattern=options.output_samples_pattern, reference=options.reference,
                  pseudo_count=options.pseudo_count)
    if shard is not None:
        results = gat_b200.runShard(segments, annotations, workspace, sampler, counters,
                                    Engine.UnconditionalWorkspace(), shard[0], shard[1], **kwargs)
    else:
        results = gat_b200.run(segments, annotations, workspace, sampler, counters,
                               workspace_generator=Engine.UnconditionalWorkspace(), **kwargs)
    if log:
        log("sampling completed in %.2f seconds" % (time.time() - t0))
    return results


def main(argv=None):
    import gat_b200
    from . import io as IO
    from . import engine as Engine
    from . import parallel

    argv = sys.argv if argv is None else argv
    parser = buildParser(usage=__doc__)
    parser.add_option("-v", "--verbose", dest="loglevel", type="int", default=1, help="log level")
    parser.add_option("-S", "--stdout", dest="stdout_file", type="string", default=None, help="output file")
    parser.add_option("--sample-range", dest="sample_range", type="string", default=None,
                      help="BEGIN:END -- sample only the global samples [BEGIN, END) of the run and write them to "
                           "--output-shard (needs --random-seed); merge the shards with python -m gat_b200.shards")
    parser.add_option("--output-shard", dest="output_shard", type="string", default=None,
                      help="shard file written by a --sample-range job")
    options, _ = parser.parse_args(argv[1:])
    shard = _shardOption(options)
    parallel.init_from_env()
    import os
    if os.environ.get("GATB_TRANSPORT", "peer") == "nccl":
        parallel.warm_up_async()        # NCCL's set-up runs behind the parsing of the input files
    rank, _ = parallel.rank_world()

    def log(msg):
        if options.loglevel >= 1 and rank == 0:
            sys.stderr.write("# %s INFO %s\n" % (time.strftime("%Y-%m-%d %H:%M:%S"), msg))

    options.stdout = open(options.stdout_file, "w") if options.stdout_file else sys.stdout
    description_header, descriptions, description_width = IO.readDescriptions(options)
    if not options.counters:
        options.counters.append("nucleotide-overlap")
    for name in ("output_tables_pattern", "output_samples_pattern", "output_counts_pattern"):
        v = getattr(options, name)
        if v is not None and "%s" not in v:
            raise ValueError("%s should contain at least one '%%s'" % name)
    if options.random_seed is not None:
        random.seed(options.random_seed)
        np.random.seed(options.random_seed)
        Engine.seed(options.random_seed)
    if options.null != "default":
        raise NotImplementedError("--null is read by the reference from a results table; pass `reference` to run()")
    options.reference = None

    if shard is not None:
        fromSegments(options, log, shard)
        if options.stdout_file:
            options.stdout.close()
        parallel.finalize()
        return 0
    if options.input_filename_counts:
        results = gat_b200.fromCounts(options.input_filename_counts)
    else:
        results = fromSegments(options, log)
    if options.pvalue_method != "empirical":
        Engine.updatePValues(results, options.pvalue_method)
    if rank == 0:
        t0 = time.time()
        IO.outputResults(results, options, Engine.AnnotatorResultExtended.headers, description_header,
                         description_width, descriptions)
        log("output written in %.2f seconds" % (time.time() - t0))
    if options.stdout_file:
        options.stdout.close()
    parallel.finalize()
    return 0


def _shardOption(options):
    """--sample-range / --output-shard -> None or ((begin, end), filename)"""
    if options.sample_range is None and options.output_shard is None:
        return None
    if options.sample_range is None or options.output_shard is None:
        raise ValueError("--sample-range and --output-shard go together")
    if options.random_seed is None:
        raise ValueError("--sample-range needs --random-seed: every shard of a run must place the same samples")
    if options.input_filename_counts:
        raise ValueError("--sample-range samples the run: it cannot start from --input-counts-file")
    try:
        begin, end = (int(x) for x in options.sample_range.split(":"))
    except ValueError:
        raise ValueError("--sample-range must be BEGIN:END, got %r" % options.sample_range)
    return (begin, end), options.output_shard


if __name__ == "__main__":
    sys.exit(main())
