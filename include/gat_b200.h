/*
 * gat_b200.h -- C ABI of the B200-native GAT simulation engine (libgat_b200.so).
 *
 * This is the drop-in boundary for the one hot path this repository accelerates: per-sample random
 * placement of segments into the workspace (SamplerAnnotator) and overlap counting of every simulated
 * set against every annotation track (Counter*), plus observed counts and per-column statistics.
 * The reference (AndreasHeger/gat 1.3.6, Python + Cython) has no FFI of its own for this path: its
 * operator interface is three duck-typed Python protocols consumed by gat.run().  Every entry point
 * below names the reference interface it replaces (paths relative to the reference checkout);
 * INTEGRATION.md shows the ctypes stub a reference maintainer would add.
 *
 * Conventions
 *   - plain C types only; all interval lists are CSR: offs[n_lists+1] (uint64) + start[] + end[]
 *     (uint32, half-open [start,end), sorted, normalized -- what SegmentList.normalize() produces,
 *     gat/SegmentList.pyx:697-754).  Coordinates must be < 2^31 (the reference's own arithmetic is
 *     int32, gat/SegmentList.pxd:31-38).
 *   - every function returns GATB_OK (0) or a negative error code; gatb_last_error() gives the text.
 *     No exceptions cross the boundary.  There is NO CPU fallback: without a CUDA device every
 *     compute entry point fails with GATB_ERR_CUDA.
 *   - one context per GPU; calls on one context are serialised by the caller; work is enqueued on
 *     the context's CUDA stream (gatb_set_stream) and entry points that return host data
 *     synchronise that stream before returning.
 *   - "host" pointers are ordinary (ideally pinned) host memory, "dev" pointers are device memory
 *     of the context's GPU (e.g. torch tensors' data_ptr()).
 */
#ifndef GAT_B200_H
#define GAT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GATB_VERSION 100

/* error codes */
#define GATB_OK              0
#define GATB_ERR_INVALID    -1   /* bad argument / inconsistent shapes                                */
#define GATB_ERR_CUDA       -2   /* CUDA runtime error (no device, launch failure, out of memory)     */
#define GATB_ERR_CAPACITY   -3   /* a placement unit overflowed its segment buffer                    */
#define GATB_ERR_TOO_LARGE  -4   /* segment too large for nbuckets*bucket_size (ValueError in         */
                                 /* SegmentList.getLengthDistribution, gat/SegmentList.pyx:1170-1182) */
#define GATB_ERR_RANGE      -5   /* coordinate >= 2^31 or total overlap >= 2^32; a histogram value outside its window */

/* counters (gat/Engine.pyx:1412-1472; names are the --counter choices, gat/__init__.py:214-223) */
#define GATB_NUCLEOTIDE_OVERLAP    0   /* CounterNucleotideOverlap       :1417-1425 */
#define GATB_NUCLEOTIDE_DENSITY    1   /* CounterNucleotideDensity       :1427-1441 */
#define GATB_SEGMENT_OVERLAP       2   /* CounterSegmentOverlap          :1443-1448 */
#define GATB_SEGMENT_MIDOVERLAP    3   /* CounterSegmentMidpointOverlap  :1450-1456 */
#define GATB_ANNOTATION_OVERLAP    4   /* CounterAnnotationOverlap       :1458-1463 */
#define GATB_ANNOTATION_MIDOVERLAP 5   /* CounterAnnotationMidpointOverlap :1465-1472 */
#define GATB_OVERLAP_PIECES        6   /* not a --counter: len(a.intersect(b)) for normalized lists = number of
                                        * overlapping (segment, interval) pairs; with nucleotide-overlap (= its
                                        * .sum()) it gives AnnotatorResultExtended's overlap_nsegments / overlap_size
                                        * columns (gat/Engine.pyx:1911-1928) for every annotation in one call */
#define GATB_NCOUNTERS             7

typedef struct gatb_ctx gatb_ctx;           /* one GPU + one stream                                  */
typedef struct gatb_annotations gatb_annotations;   /* annotation tracks staged for counting         */
typedef struct gatb_sampler gatb_sampler;   /* one segment track + workspace staged for placement    */

/* ---- context ----------------------------------------------------------------------------------*/
int         gatb_version(void);
int         gatb_create(int device, gatb_ctx **out);
void        gatb_destroy(gatb_ctx *ctx);
const char *gatb_last_error(gatb_ctx *ctx);            /* ctx may be NULL: last creation error       */
/* cuda_stream: a cudaStream_t; NULL selects the context's own (non-blocking) stream.  A caller that works on the
 * legacy default stream -- e.g. PyTorch's default stream, whose handle is 0 -- passes cudaStreamLegacy ((void *)1),
 * otherwise the library's work would not be ordered with the caller's. */
int         gatb_set_stream(gatb_ctx *ctx, void *cuda_stream);
int         gatb_synchronize(gatb_ctx *ctx);
/* number of this library's kernels launched on the context since creation (bench "gpu_launches") */
uint64_t    gatb_launch_count(gatb_ctx *ctx);

/* optional per-kernel timing: when enabled, every kernel launch is bracketed by CUDA events on the
 * context's stream.  gatb_profile_read synchronises and returns (and clears) the accumulated device
 * milliseconds and launch counts per kernel class: [0] placement K1, [1] isochore merge K2,
 * [2] counting K3/K4, [3] everything else (preparation, tally, statistics). */
int         gatb_profile(gatb_ctx *ctx, int enable);
int         gatb_profile_read(gatb_ctx *ctx, double *ms /*[4]*/, uint64_t *launches /*[4]*/);

/* ---- annotations ------------------------------------------------------------------------------
 * Replaces the `contig_annotations` IntervalCollection that UnconditionalSampler.sample() hands to
 * every computeSample() call (gat/__init__.py:716-718, :580-587), flattened: n_annot tracks x n_keys
 * keys (contigs for sampling, "contig.isochore" keys for observed counts), annotation-major:
 * list (a, k) = [offs[a*n_keys+k], offs[a*n_keys+k+1]).  key_ws_nseg[k] = len(workspace[key])
 * (number of workspace SEGMENTS, the nucleotide-density denominator, gat/Engine.pyx:1437-1441);
 * may be NULL when density is never requested.  Host pointers; data is copied to the device. */
int  gatb_annotations_create(gatb_ctx *ctx, int n_annot, int n_keys, const uint64_t *offs,
                             const uint32_t *start, const uint32_t *end, const uint32_t *key_ws_nseg,
                             gatb_annotations **out);
/* The same without waiting: the copies and the index build are queued on a separate upload stream and
 * the call returns; the first gatb_run / gatb_count_lists using the set waits for them (gatb_run
 * only after it has queued its first placement kernel, so upload and build overlap the placement) and
 * reports a failed validation (GATB_ERR_INVALID / GATB_ERR_RANGE) when it returns.  offs / start / end
 * must stay valid and unchanged until that call or gatb_annotations_wait() has returned; pinned host
 * memory makes the copies truly asynchronous.  gatb_annotations_wait blocks until the set is built and
 * returns the validation result; a failed set can only be destroyed. */
int  gatb_annotations_create_async(gatb_ctx *ctx, int n_annot, int n_keys, const uint64_t *offs,
                                   const uint32_t *start, const uint32_t *end, const uint32_t *key_ws_nseg,
                                   gatb_annotations **out);
int  gatb_annotations_wait(gatb_annotations *a);
void gatb_annotations_destroy(gatb_annotations *a);

/* ---- input preparation on the device ---------------------------------------------------------------
 * Interval lists resident on the GPU as CSR (gatb_lists): what IO.buildSegments / IO.applyIsochores do to a large
 * collection with per-list host loops (gat/IO.py:88-293) runs as a few sorts and scans over ALL lists at once, and
 * the annotation set is built from the result without the intervals ever returning to the host.
 *   gatb_lists_from_rows     rows (list_id, start, end) in any order -> sorted lists with overlapping rows merged:
 *                            join_adjacent 0 = IntervalCollection.normalize() / SegmentList.normalize
 *                            (gat/Engine.pyx:2941-2956, gat/SegmentList.pyx:697-754: adjacent segments stay apart),
 *                            1 = merge(0) (:756-816: adjacent segments join).  Empty rows (start == end) vanish.
 *   gatb_lists_from_csr      lists that are already normalized on the host (the workspace, the isochore tracks)
 *   gatb_lists_restrict      list l of `in` (n_tracks x n_keys lists, key = l % n_keys) against the `fanout` lists
 *                            other[key * fanout + f]: truncate != 0 -> SegmentList.intersect (gat/SegmentList.pyx:
 *                            1469-1549), else SegmentList.filter (:1401-1467); the result has in.n_lists * fanout
 *                            lists, list l * fanout + f.  fanout 1 with the workspace = annotations.intersect(workspace)
 *                            (gat/IO.py:232-236); fanout = number of isochore tracks = toIsochores (gat/Engine.pyx:
 *                            2837-2855, gat/IO.py:201-210).
 *   gatb_lists_collapse      every `fanout` consecutive lists extended into one, then merge(0):
 *                            IntervalDictionary.fromIsochores (gat/Engine.pyx:2857-2876)
 *   gatb_lists_select        new lists out[l] = in[src[l]] (src[l] >= in.n_lists: an empty list): the key order of
 *                            another dictionary
 *   gatb_lists_sizes         len() and sum() of every list (host arrays, n_lists each; either may be NULL)
 *   gatb_lists_download      the CSR arrays to the host (offs[n_lists + 1], start / end[n_intervals]; any may be NULL)
 *   gatb_annotations_create_from_lists   gatb_annotations_create reading n_annot x n_keys device lists in place */
typedef struct gatb_lists gatb_lists;
int  gatb_lists_from_rows(gatb_ctx *ctx, uint64_t n_rows, const uint32_t *list_id, const uint32_t *start,
                          const uint32_t *end, uint32_t n_lists, int join_adjacent, gatb_lists **out);
int  gatb_lists_from_csr(gatb_ctx *ctx, uint32_t n_lists, const uint64_t *offs, const uint32_t *start,
                         const uint32_t *end, gatb_lists **out);
int  gatb_lists_restrict(const gatb_lists *in, uint32_t n_keys, uint32_t fanout, const gatb_lists *other,
                         int truncate, gatb_lists **out);
int  gatb_lists_collapse(const gatb_lists *in, uint32_t fanout, gatb_lists **out);
int  gatb_lists_select(const gatb_lists *in, uint32_t n_out, const uint32_t *src, gatb_lists **out);
int  gatb_lists_info(const gatb_lists *lists, uint32_t *n_lists, uint64_t *n_intervals);
int  gatb_lists_sizes(const gatb_lists *lists, uint64_t *count, uint64_t *bases);
int  gatb_lists_download(const gatb_lists *lists, uint64_t *offs, uint32_t *start, uint32_t *end);
void gatb_lists_destroy(gatb_lists *lists);
int  gatb_annotations_create_from_lists(gatb_ctx *ctx, const gatb_lists *lists, int n_annot, int n_keys,
                                        const uint32_t *key_ws_nseg, gatb_annotations **out);

/* ---- counting of given (placed or observed) segment sets ----------------------------------------
 * Replaces, for n_samples segment sets at once, the loop
 *     counts[counter][annotation] = sum(counter(sample[key], annotations[annotation][key],
 *                                               workspace[key]) for key in sample.keys())
 * of computeSample (gat/__init__.py:580-587) and of Engine.computeCounts (gat/Engine.pyx:2189-2202).
 * Sample s, key k owns the list [offs[s*n_keys+k], offs[s*n_keys+k+1]) of start/end (host pointers).
 * key_present[s*n_keys+k] (may be NULL = all present) says whether the key is in sample.keys():
 * absent keys add nothing, present-but-empty keys add 0 (only visible in float rounding).
 * counters[n_counters] lists counter ids; out is host memory, [n_counters][n_samples][n_annot]
 * doubles (integers are exact in a double; nucleotide-density is the float64 sum in key order). */
int  gatb_count_lists(gatb_ctx *ctx, const gatb_annotations *annos, int n_counters, const int32_t *counters,
                      uint64_t n_samples, const uint64_t *offs, const uint32_t *start, const uint32_t *end,
                      const uint8_t *key_present, double *out);

/* ---- placement --------------------------------------------------------------------------------
 * Replaces SamplerAnnotator(bucket_size, nbuckets).sample(segments[key], workspace[key]) for every
 * key of one segment track (gat/Engine.pyx:502-646, called from gat/__init__.py:531-546).
 * Units are the keys of the track in iteration order, already skipping keys whose segment list or
 * workspace is empty (gat/__init__.py:536-538).  unit_contig[u] in [0,n_contigs) is the contig the
 * key belongs to ("contig.iso".split(".")[0], gat/Engine.pyx:2863-2866), contigs numbered in order of
 * first appearance (= sample.keys() order after fromIsochores); has_isochores != 0 when keys carry an
 * isochore suffix, in which case each contig's placed lists are concatenated and merge(0)-ed before
 * counting (gat/Engine.pyx:2857-2876).  bucket_size / nbuckets as in --bucket-size / --nbuckets
 * (bucket_size 0 = automatic, gat/SegmentList.pyx:1164-1165; GATB_ERR_TOO_LARGE where getLengthDistribution
 * raises "segment too large", :1170).  nbuckets = 0 builds NO length histogram: such a sampler serves
 * gatb_sampler_set_shift only -- SamplerShift never calls getLengthDistribution (gat/Engine.pyx:1060-1062),
 * so no segment is too large for it.  Host pointers; data is copied to the device and
 * the sample-invariant preparation (filter, ltotal, length table, workspace CDF: gat/Engine.pyx:543-565)
 * runs once, on the GPU. */
int  gatb_sampler_create(gatb_ctx *ctx, int n_units, const int32_t *unit_contig, int n_contigs,
                         int has_isochores,
                         const uint64_t *seg_offs, const uint32_t *seg_start, const uint32_t *seg_end,
                         const uint64_t *ws_offs, const uint32_t *ws_start, const uint32_t *ws_end,
                         uint32_t bucket_size, uint32_t nbuckets, gatb_sampler **out);
void gatb_sampler_destroy(gatb_sampler *s);
/* capacity (in segments) of one sample's contig-level output (gatb_sampler_place) and of its unit-level
 * output (gatb_sampler_place_units).  Capacities are estimates made at creation; a unit that outgrows its
 * buffer is grown by the library and the call repeated internally (the reference's lists grow on demand,
 * gat/SegmentList.pyx:513-537), after which these values are larger. */
uint64_t gatb_sampler_sample_capacity(const gatb_sampler *s);
uint64_t gatb_sampler_unit_capacity(const gatb_sampler *s);

/* Sampler used for placement: 0 = SamplerAnnotator (default), 1 = SamplerSegments (gat/Engine.pyx:653-737:
 * exactly len(segments[key]) placements per unit, all kept).  SamplerSegments' samples are unsorted and
 * overlapping; they are only normalized by fromIsochores' merge(0), so kind 1 requires has_isochores
 * (without it the reference's counters fail their isNormalized assertion). */
int  gatb_sampler_set_kind(gatb_sampler *s, int kind);

/* Sampler kind 2 = SamplerShift(radius, extension) (gat/Engine.pyx:998-1111; gat-run.py --sampler=shift
 * --shift-expansion=radius --shift-extension=extension, scripts/gat-run.py:129-132): every segment that
 * overlaps its unit's workspace moves to a random workspace position within floor(length * radius / 2)
 * bases (or extension / 2 when extension != 0) of its midpoint, wrapped around the ends of that local
 * workspace; the sample is normalized per unit (adjacent pieces stay apart) and, with isochores, merged per
 * contig.  Works with and without isochores.  Re-sizes the sampler's buffers (eight pieces per segment); a
 * unit whose moved segments are cut into more pieces makes gatb_run / gatb_sampler_place return
 * GATB_ERR_CAPACITY.  A segment whose window holds no workspace drops out of the sample, as in the
 * reference (where getRandomPosition's ValueError is printed and ignored).  Needs length * radius / 2 < 2^31. */
int  gatb_sampler_set_shift(gatb_sampler *s, double radius, int32_t extension);

/* Place samples [sample_begin, sample_begin+n_samples) and return the contig-level segment sets
 * (what `sample` holds after sample.fromIsochores(), gat/__init__.py:563) to the host:
 * counts[s*n_contigs+c] segments for contig c of sample s, stored at start/end[s*capacity + contig_base[c] ...]
 * where capacity = gatb_sampler_sample_capacity() and contig_base is returned in contig_base[n_contigs].
 * unit_status[s*n_units+u] (may be NULL): bit0 = stopped after 20 non-improving rounds
 * (gat/Engine.pyx:570-572), bit1 = capacity overflow.  For tests and the same-placement parity fixture.
 * GATB_ERR_CAPACITY: a unit outgrew its buffer and the library enlarged it -- the arrays sized from the
 * earlier capacity query are too small: query gatb_sampler_sample_capacity() again and repeat the call. */
int  gatb_sampler_place(gatb_sampler *s, uint64_t seed, uint32_t track, uint64_t sample_begin,
                        uint64_t n_samples, uint32_t *start, uint32_t *end, uint32_t *counts,
                        uint64_t *contig_base, uint8_t *unit_status);

/* The same placement, returned per UNIT (= per key of the track, "contig" or "contig.isochore"), before
 * fromIsochores: exactly what sampler.sample(segs[key], workspace[key]) returns for every key
 * (gat/__init__.py:531-546) and what --output-samples-pattern writes under each key (:518-559).  For
 * SamplerSegments (kind 1) the lists are in draw order, unsorted and unmerged (gat/Engine.pyx:719-735).
 * counts[s*n_units+u] segments of unit u of sample s at start/end[s*capacity + unit_base[u] ...] with
 * capacity = gatb_sampler_unit_capacity(); GATB_ERR_CAPACITY as for gatb_sampler_place. */
int  gatb_sampler_place_units(gatb_sampler *s, uint64_t seed, uint32_t track, uint64_t sample_begin,
                              uint64_t n_samples, uint32_t *start, uint32_t *end, uint32_t *counts,
                              uint64_t *unit_base, uint8_t *unit_status);

/* ---- the hot path: place + count ----------------------------------------------------------------
 * Replaces UnconditionalSampler.sample() (gat/__init__.py:704-778) for one track: for every sample
 * in [sample_begin, sample_begin+n_samples) place all units, merge per contig, count against every
 * annotation with every requested counter.  The random stream is keyed by (seed, track, unit,
 * GLOBAL sample index, turn), so the result does not depend on how samples are sharded over GPUs.
 *   out_counts: [n_counters][n_samples][n_annot]; uint32 for the integer counters, and the
 *   nucleotide-density plane (if requested) is float64 stored in out_density[n_samples][n_annot].
 *   out_is_device != 0: out_counts / out_density are device pointers (results stay in HBM, no sync);
 *   otherwise host pointers (copied back, stream synchronised).
 *   info (may be NULL, host): [0] total segments placed (contig level), [1] units that hit the
 *   20-round cap, [2] 0.  A unit that outgrows its buffer is grown and the call runs again internally
 *   (same stream of draws, hence the same result as a run with enough room from the start);
 *   GATB_ERR_CAPACITY only if one contig needed more than 2^24 slots. */
int  gatb_run(gatb_sampler *s, const gatb_annotations *annos, int n_counters, const int32_t *counters,
              uint64_t seed, uint32_t track, uint64_t sample_begin, uint64_t n_samples,
              uint32_t *out_counts, double *out_density, int out_is_device, uint64_t *info);
/* samples placed + counted per internal batch (memory/parallelism knob; 0 = default) */
int  gatb_set_batch_size(gatb_ctx *ctx, uint32_t batch);

/* ---- multi-GPU exchange fused into the counting kernel --------------------------------------------------
 * Samples are independent (gat/__init__.py:738-747, the results are only concatenated :770-774): rank g of G
 * computes its shard of the global sample indices and the S x A count matrix is assembled from the shards.
 * Instead of a collective AFTER the kernels, gatb_run can deliver every finished row to several destinations at
 * once -- OUTPUT ROUTES: route r receives the columns
 * [col_begin, col_end) of counter plane c, sample row s at
 *     base + c * plane_stride + (row0 + s) * row_stride + (annotation - col_begin)         (uint32 elements)
 * where s counts from the call's sample_begin.  `base` may be memory of another GPU of the box, mapped with
 * gatb_peer_open over NVLink / NVSwitch: all columns to every rank's [S][A] matrix is the all-gather of the
 * sample slabs; every rank's own column block to its [S][A_g] matrix is the all-to-all by column (column-sharded
 * statistics).  The caller synchronises the ranks (any barrier) after the last gatb_run before reading.
 * Routes stay set until replaced (n_routes = 0 clears them); with routes, gatb_run takes integer counters only; with
 * out_is_device != 0 it ignores out_counts, with host outputs the rows go to the host matrix AND to the routes.
 * Two ways to serve the routes (gatb_set_route_mode; same results): by_kernel = 0 (default) -- the kernel writes a
 * staging slab and COPY ENGINES scatter its rows / column blocks to the routes (2-D device-to-device copies on a copy
 * stream, peer GPUs included) while the next batch is already being placed and counted; by_kernel = 1 -- the counting
 * kernel's epilogue stores every row to every route itself (no staging, no copies; its NVLink stores sit at the end of
 * the kernel where nothing overlaps them: measured 4 % slower per step on 8 GPUs).
 * Peer memory: gatb_peer_alloc allocates shareable device memory and returns its 64-byte IPC handle (send it to
 * the other processes by any means), gatb_peer_open maps another process's allocation into this one. */
#define GATB_PEER_HANDLE_BYTES 64
typedef struct gatb_route {
    uint32_t *base;
    uint64_t plane_stride;          /* elements between counter planes */
    uint64_t row_stride;            /* elements between sample rows */
    uint64_t row0;                  /* row of the call's first sample */
    uint32_t col_begin, col_end;    /* annotation columns delivered */
} gatb_route;
int  gatb_set_output_routes(gatb_ctx *ctx, int n_routes, const gatb_route *routes);
int  gatb_set_route_mode(gatb_ctx *ctx, int by_kernel);
int  gatb_peer_alloc(gatb_ctx *ctx, uint64_t bytes, void **ptr, unsigned char *handle /*[64]*/);
int  gatb_peer_free(gatb_ctx *ctx, void *ptr);
int  gatb_peer_open(gatb_ctx *ctx, const unsigned char *handle /*[64]*/, void **ptr);
int  gatb_peer_close(gatb_ctx *ctx, void *ptr);

/* ---- measurement aids (bench.py `roofline`; no reference counterpart) ------------------------------
 * gatb_count_work: the work of the counting kernel on the LAST internal batch of the preceding gatb_run on
 * this sampler (n_samples = size of that batch): out[0] placed segments, out[1] index entries in their runs
 * (= entries the kernel tests, padding included; compare with the truly overlapping pairs given by the
 * GATB_OVERLAP_PIECES counter), out[2] entries of the whole index, out[3] bytes of the index arrays read.
 * gatb_microbench: a machine peak measured on `device` with CUDA events, best of `repeats` runs:
 *   which 0: L2 read bandwidth (a `bytes`-sized buffer, default 48 MB, streamed by every SM with 16-byte
 *            loads) -> out[0] GB/s;   which 1: warp-instruction issue rate (interleaved integer and FP32
 *            chains on 64 warps per SM) -> out[0] 1e9 warp instructions/s.   out[1] ms of the best run, out[2] its work
 *            (bytes / warp instructions), out[3] number of SMs. */
int  gatb_count_work(gatb_sampler *s, const gatb_annotations *annos, uint32_t n_samples, uint64_t *out /*[4]*/);
int  gatb_microbench(int device, int which, uint64_t bytes, int repeats, double *out /*[4]*/);

/* ---- per-column statistics ------------------------------------------------------------------------
 * Replaces makeEnrichmentStatistics + getTwoSidedPValue (gat/Engine.pyx:1635-1718, :1543-1576) for
 * n_cols columns of n_samples simulated counts each: expected (numpy.mean), stddev (numpy.std, ddof 0),
 * CI95 low/high (sorted[min(off,l-1)], sorted[max(l-off,0)], off=int(0.05*l)), fold with pseudo-count,
 * empirical two-sided p-value.  counts is [n_samples][n_cols] uint32 (is_float==0) or float64
 * (is_float!=0), device memory if counts_is_device else host.  observed[n_cols], ref_fold[n_cols]
 * (NULL = no --null reference) and all outputs are host arrays of n_cols doubles.
 * uint32 matrices are reduced with integer arithmetic only (sum, 128-bit sum of squares, counts, radix select): every
 * output but stddev is exact, stddev is the correctly rounded sqrt((n*sum x^2 - (sum x)^2) / n^2) -- within a few ulp
 * of numpy.std -- and no output depends on the GPU, the grid or on which other columns share the matrix. */
int  gatb_column_stats(gatb_ctx *ctx, const void *counts, int is_float, int counts_is_device,
                       uint64_t n_samples, int n_cols, const double *observed, const double *ref_fold,
                       double pseudo_count, double *expected, double *stddev, double *lower95,
                       double *upper95, double *fold, double *pvalue);

/* Replaces AnnotatorResult.getEmpiricalPValue(value) (gat/Engine.pyx:1829-1831 -> getTwoSidedPValue,
 * :1543-1576): the two-sided empirical p-value of values[a] among the samples of column a, where the over- /
 * under-representation branch is chosen against the result's STORED expectation expected[a] (which includes a
 * --null reference fold, :1673-1676).  counts as in gatb_column_stats; values, expected, pvalue: host, n_cols. */
int  gatb_column_pvalue(gatb_ctx *ctx, const void *counts, int is_float, int counts_is_device,
                        uint64_t n_samples, int n_cols, const double *values, const double *expected,
                        double *pvalue);

/* ---- per-column statistics without the sample matrix ----------------------------------------------
 * Replaces makeEnrichmentStatistics + getTwoSidedPValue (gat/Engine.pyx:1635-1718, :1543-1576) like
 * gatb_column_stats, for a uint32 counter plane [n_samples_total][n_cols] that is never held whole: the rows
 * arrive as slabs in device memory (e.g. what gatb_run writes with out_is_device), are counted and may then be
 * overwritten.  The accumulator keeps exact integers per column -- sum, 128-bit sum of squares, #{x < observed},
 * #{x == observed}, smallest and largest value -- plus, for the two CI95 order statistics, a window of unit-width
 * uint32 bins [lo[a], lo[a] + width[a]) per column and the counts below / above it.  Integers add across slabs (and
 * across ranks, gatb_colacc_state / gatb_colacc_merge), so for every column whose two CI ranks fall inside its
 * window gatb_colacc_finish returns exactly the doubles gatb_column_stats returns for the whole matrix.  A column
 * whose rank falls outside ("missed") needs its histogram again with a wider window ([min, max] of the column
 * always holds it): set new windows and add the same rows once more with GATB_COLACC_HIST only. */
typedef struct gatb_colacc gatb_colacc;
#define GATB_COLACC_SUMS 1   /* gatb_colacc_add: count the rows into the sums (each row of the plane once)    */
#define GATB_COLACC_HIST 2   /*                  count the rows into the windows' histograms                 */

/* observed[n_cols], ref_fold[n_cols] (NULL = no --null reference): host, as in gatb_column_stats;
 * 1 <= n_samples_total < 2^32.  Every column starts with an empty window (every value counts as above it). */
int  gatb_colacc_create(gatb_ctx *ctx, int n_cols, uint64_t n_samples_total, const double *observed,
                        const double *ref_fold, gatb_colacc **out);
/* lo[n_cols], width[n_cols] (host): the windows; clears the histograms (and below / above), keeps the sums.  The
 * bins of all columns live in one device arena of sum(width) uint32 (lo + width <= 2^32). */
int  gatb_colacc_set_windows(gatb_colacc *acc, const uint32_t *lo, const uint32_t *width);
/* counts (dev): n_rows rows of n_cols uint32, row_stride (>= n_cols) elements apart.  what: GATB_COLACC_SUMS
 * and/or GATB_COLACC_HIST.  Enqueued on the context's stream, no synchronisation: the slab may be reused by
 * work enqueued after it on that stream. */
int  gatb_colacc_add(gatb_colacc *acc, const uint32_t *counts, uint64_t n_rows, uint64_t row_stride, int what);
/* the integer state, host arrays, any of them NULL: rows counted into the sums, moments [5][n_cols] (sum,
 * #{x < observed}, #{x == observed}, sum x^2 low 64 bits, high 64 bits), minmax [2][n_cols], outside [2][n_cols]
 * (below, above), bins [sum(width)]. */
int  gatb_colacc_state(gatb_colacc *acc, uint64_t *rows, uint64_t *moments, uint32_t *minmax, uint64_t *outside,
                       uint32_t *bins);
/* adds another accumulator's state (same columns, observed values and windows; gatb_colacc_state layout) into
 * this one: the sum of squares with its carry, min / max, counts. */
int  gatb_colacc_merge(gatb_colacc *acc, uint64_t rows, const uint64_t *moments, const uint32_t *minmax,
                       const uint64_t *outside, const uint32_t *bins);
/* the windows' histograms as sparse CSR, compacted on the device (a per-column count of the non-zero bins, a scan, an
 * emit pass): col_ptr[n_cols + 1] (host) receives the offsets, and entries col_ptr[a] .. col_ptr[a + 1] - 1 of value /
 * count (host, `capacity` entries) the non-zero bins of column a in increasing value.  Two calls, as
 * gatb_format_counts: value == count == NULL asks for col_ptr only (col_ptr[n_cols] = entries needed);
 * GATB_ERR_CAPACITY when capacity is too small (col_ptr is still filled). */
int  gatb_colacc_export(gatb_colacc *acc, int64_t *col_ptr, uint32_t *value, uint64_t *count, uint64_t capacity);
/* adds a sparse histogram (gatb_colacc_export layout, host arrays, col_ptr[n_cols] entries) into the windows' bins:
 * count[i] at value[i] of its column.  GATB_ERR_RANGE, with the bins untouched, when a value lies outside its
 * column's window or a count is 2^32 or more.  Enqueued on the context's stream after the check. */
int  gatb_colacc_add_sparse(gatb_colacc *acc, const int64_t *col_ptr, const uint32_t *value, const uint64_t *count);
/* the statistics of gatb_column_stats (host outputs of n_cols doubles, any may be NULL) once the sums hold
 * n_samples_total rows and every histogram n_samples_total values (GATB_ERR_INVALID otherwise).  missed[n_cols]
 * (host, may be NULL): 1 where a CI rank fell outside the column's window -- lower95 / upper95 are NaN there,
 * every other output is exact. */
int  gatb_colacc_finish(gatb_colacc *acc, double pseudo_count, double *expected, double *stddev, double *lower95,
                        double *upper95, double *fold, double *pvalue, uint8_t *missed);
void gatb_colacc_destroy(gatb_colacc *acc);

/* ---- gat-compare: pairwise comparison of fold changes ----------------------------------------------
 * Replaces the inner loop of scripts/gat-compare.py (:218-241 within one counts file, :300-323 between
 * two): for pair q of columns (col1[q] of m1, col2[q] of m2)
 *     fc1 = obs1[q] / (m1[:, col1[q]] + pseudo_count) + 1e-4,   fc2 likewise
 *     sampled = log(fc1 / fc2) + delta[q]            (delta = fold2 - fold1, the observed value)
 *     AnnotatorResult(observed = delta[q], samples = sampled, pseudo_count = 0)
 * i.e. the column statistics of gatb_column_stats on the derived samples, which never leave the GPU.
 * m1 / m2: host, [n_samples][n_cols] float64 (m2 may equal m1); all other arrays host, n_pairs long. */
int  gatb_compare_stats(gatb_ctx *ctx, uint64_t n_samples, const double *m1, int n_cols1,
                        const double *m2, int n_cols2, uint64_t n_pairs, const int32_t *col1,
                        const int32_t *col2, const double *obs1, const double *obs2, const double *delta,
                        double pseudo_count, double *expected, double *stddev, double *lower95,
                        double *upper95, double *fold, double *pvalue);
/* gatb_compare_stats on DEVICE matrices: m1 / m2 [n_samples][n_cols] each uint32, or float64 where is_float (m2 may
 * equal m1); all other arrays host, as above.  A uint32 converted to double is exact, so every output is bit-identical
 * to gatb_compare_stats on the same values stored as float64. */
int  gatb_compare_stats_device(gatb_ctx *ctx, uint64_t n_samples, const void *m1, int is_float1, int n_cols1,
                               const void *m2, int is_float2, int n_cols2, uint64_t n_pairs, const int32_t *col1,
                               const int32_t *col2, const double *obs1, const double *obs2, const double *delta,
                               double pseudo_count, double *expected, double *stddev, double *lower95,
                               double *upper95, double *fold, double *pvalue);

/* ---- counts table: the text of --output-counts-pattern ------------------------------------------------
 * Replaces the Python loop of gat/__init__.py:1072-1086, which writes for every result
 *     ",".join(["%i" % x for x in samples])
 * (2e8 numbers at 1e6 samples x 200 annotations).  For an [n_samples][n_cols] uint32 count matrix (host, or
 * device with counts_is_device) the decimal text of every COLUMN, comma separated, no trailing separator, is
 * formatted on the GPU.  col_off[n_cols + 1] (host) receives the byte offset of every column's text;
 * text (host, `capacity` bytes) receives the bytes and may be NULL to ask for the sizes only
 * (col_off[n_cols] = bytes needed).  GATB_ERR_CAPACITY when capacity is too small (col_off is still filled). */
int  gatb_format_counts(gatb_ctx *ctx, const uint32_t *counts, int counts_is_device, uint64_t n_samples,
                        int n_cols, uint64_t *col_off, char *text, uint64_t capacity);

/* ---- counts table reader: --input-counts-file and gat-compare -------------------------------------------
 * Replaces the Python loop of gat/__init__.py:1091-1119, which parses every number of a counts table with
 *     numpy.array(list(map(float, counts.split(","))))
 * text (device, n_bytes): the BODY of a table, the bytes after its header line.  Plain = every line is
 *     field \t field \t field \t D(,D)* \n
 * with D = 1 to 10 ASCII digits of value <= 2^32 - 1 (leading zeros allowed), the same number of D on every line,
 * the last byte '\n' and no '\r' anywhere.  Line r is column r of the uint32 matrix counts[n_samples][n_rows] (the
 * layout of gatb_column_stats).  Two calls, as gatb_format_counts:
 *   counts == NULL: *n_rows, *n_samples, *plain and *bad_offset, the offset of the first byte outside the grammar
 *       (UINT64_MAX when plain; for a line with fewer values than the first line, its '\n', for one with more, its first
 *       extra comma), and for a
 *       plain table lines[2 * r] = start of line r, lines[2 * r + 1] = start of its counts field (host, line_capacity
 *       pairs; GATB_ERR_CAPACITY when there are more lines, the counts are still returned)
 *   counts != NULL (device, n_samples * n_rows uint32, caller-allocated): the same, and the matrix; GATB_ERR_INVALID
 *       when the text is not plain.
 * An empty body is plain with no rows. */
int  gatb_parse_counts(gatb_ctx *ctx, const char *text, uint64_t n_bytes, uint64_t line_capacity, uint64_t *n_rows,
                       uint64_t *n_samples, int *plain, uint64_t *bad_offset, uint64_t *lines, uint32_t *counts);

#ifdef __cplusplus
}
#endif
#endif /* GAT_B200_H */
