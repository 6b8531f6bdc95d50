// count.cuh -- counting kernel (K3/K4), the annotation grid index and column statistics (K5).
//
// Replaces overlapWithSegments / intersectionWithSegments (gat/SegmentList.pyx:1026-1146) as used by
// the Counter* classes (gat/Engine.pyx:1412-1472) inside computeSample (gat/__init__.py:580-587) and
// computeCounts (gat/Engine.pyx:2189-2202).
#pragma once

#include "common.cuh"

namespace gatb {

constexpr uint32_t GROUP_TRACKS_MAX = 4096;   // annotation tracks per group (shared-memory accumulators per sample)

constexpr uint32_t ENTRY_LEN_MASK = 0xfffffu;

// Annotation index = a uniform GRID over every key (contig), shared by all tracks of a group (normally:
// all tracks).  Bin b of a key covers positions [b << shift, (b+1) << shift) and owns TWO entry lists:
//   S[b]  the intervals (of every track) that START in bin b          -- every interval exactly once
//   C[b]  the intervals that start before bin b and reach into it     -- an interval crossing m bin boundaries m times
// The S lists of a key are stored back to back in bin order, so the intervals starting anywhere in bins b0..b1 are
// ONE contiguous run.  A segment [s,e) covering bins b0..b1 meets every interval that can overlap it in exactly
// two runs -- C[b0] (started earlier, still open at the left edge of b0) and S[b0..b1] -- and meets it ONCE, so no
// de-duplication is needed: two offset pairs replace the binary search (utils/gat_utils.c:8-32) for all tracks at
// once.  Nearly every entry of C[b0] truly overlaps the segment (its interval is open at b0's left edge and only has
// to reach s); the waste is the S entries of bins b0 / b1 outside [s,e): ~W/2 bases' worth at either end.
// Entries of a list are in no particular order (built with atomics); all accumulation is by integer atomics, so
// results do not depend on it.  Every list holds an EVEN number of entries (an odd one is padded with an entry
// that overlaps nothing: start 2^31-1) and so starts on an even index: the counting kernel reads entries two at a
// time (16-byte loads) and a pair never straddles two segments' runs.
//
//   KeyBins keybins[n_groups][n_keys]    where the key's bins start in the offset arrays, how many, log2(bin width)
//   uint32  boff[2 * (n_boff + 1)]       first half: per (group, key) nbins+1 offsets of the S lists, second half
//                                        (at boff + n_boff + 1): of the C lists; absolute, into the arrays below
//                                        (all S lists first, then all C lists)
//   uint4   brec[n_boff]                 the offsets again, as the counting kernel reads them: one 16-byte record per
//                                        bin {C start, S start, |C| and |S[b]|, |S[b..b+1]| and |S[b..b+2]|} (16-bit
//                                        lengths) = ONE load per segment unless it spans more than three bins
//   uint2   cent[n_entries]              the entry the counting kernel streams, 8 bytes:
//                                          .x = start,  .y = min(length, 2^20-1)<<12 | slot
//                                        (slot = track within the group, < 4096; a length field of 2^20-1
//                                        sends the kernel to civ[] for the end)
//   uint2   civ[n_entries]               the exact interval (start, end), read for intervals of 2^20-1 bases or more
//   uint32  cprev[n_entries]             end of the previous interval of the same track on this key (0: none):
//                                        "is this the first interval of its track overlapping [s,e)?" = cprev <= s
struct KeyBins {
    uint64_t base;      // index into boff[] of the key's first offset
    uint32_t nbins;     // 0: no interval of any track of the group on this key
    uint32_t shift;     // 4 .. 20
};

// Where a count launch delivers its integer results.  Without routes: out_u32[sample][annotation].  With routes,
// every route r receives the columns [col_begin, col_end) of every sample row, at
//     base[(row0 + sample) * row_stride + (annotation - col_begin)]
// `base` may be memory of ANOTHER GPU of the box (peer-mapped over NVLink, gatb_peer_open): the kernel's epilogue
// then IS the exchange step of a multi-GPU run -- all columns to every rank = the all-gather of the sample slabs,
// each rank's own column block = the all-to-all by column -- with no collective launched afterwards.
constexpr uint32_t GATB_MAX_ROUTES = 16;
struct OutRoute {
    uint32_t *base;
    uint64_t row_stride;
    uint64_t row0;
    uint32_t col_begin, col_end;
};

struct CountParams {
    // annotations
    const KeyBins *keybins;         // [n_groups][n_keys]
    const uint32_t *boff;           // S offsets; the C offsets follow at boff + coff_base
    uint64_t coff_base;             // = n_boff + 1
    const uint4 *brec;              // the same offsets as one packed record per bin (bins_rec_kernel)
    const uint2 *cent;
    const uint2 *civ;
    const uint32_t *cprev;
    uint32_t has_long;              // the index holds intervals of >= 2^20 - 1 bases (their ends are read from civ[])
    uint32_t sentinel;              // index of the pair of entries that overlap nothing (= capacity, even; arrays hold capacity + 2)
    const uint32_t *key_ws_nseg;    // [n_keys] or NULL
    uint32_t n_annot, n_keys, n_groups, ka;   // ka = tracks per group
    uint32_t kgrp;                  // keys whose item tables are held in shared memory at a time
    // segment sets
    const uint64_t *placed;         // [n_samples][sample_stride] packed
    uint64_t sample_stride;
    const uint64_t *key_base;       // [n_keys]
    const uint32_t *placed_n;       // [n_samples][n_keys]
    const uint8_t *key_present;     // [n_samples][n_keys] or NULL
    uint32_t n_samples;
    uint32_t schunk;                // samples per CTA
    // output
    uint32_t *out_u32;              // [n_samples][n_annot] (integer counters)
    double *out_f64;                // [n_samples][n_annot] (nucleotide-density)
    uint32_t n_routes;              // > 0: the integer results go to routes[] instead of out_u32
    OutRoute routes[GATB_MAX_ROUTES];
};

// shared memory of a count launch: per-warp staging, accumulators [schunk][ka] (u32; density: + (sum,
// compensation) doubles), item tables of kgrp keys
size_t count_smem_bytes(uint32_t schunk, uint32_t ka, uint32_t kgrp, int threads, bool density);

// Builds the grid index from the raw annotation CSR arrays on the device and validates the lists
// (error bit 0: coordinate >= 2^31, bit 1: empty / unsorted / overlapping = not normalized, bit 2: more
// entries than `capacity`).  Launches: count the S and C entries per bin, round up to even, ONE exclusive scan over
// both halves of boff[] (so the C lists follow the S lists in the entry arrays), fill, pad.
struct BuildBinsParams {
    const uint64_t *offs;           // [n_annot*n_keys+1]
    const uint32_t *start, *end;
    uint64_t n_intervals;
    const KeyBins *keybins;         // [n_groups][n_keys]
    const uint32_t *key_jmax;       // [n_keys] longest list (over all tracks) on the key
    uint32_t jmax_all;              // largest of them
    uint4 *brec;                    // [n_boff] out: per-bin records for the counting kernel
    uint32_t *boff;                 // [2 * (n_boff + 1)], zeroed by the caller: S half, then C half
    uint64_t n_boff;                // offset slots of one half: sum over (group, key) of nbins + 1
    uint2 *cent;
    uint2 *civ;
    uint32_t *cprev;
    uint64_t capacity;              // entries the arrays hold (even), + 2 for the sentinel pair
    uint32_t n_annot, n_keys, n_groups, ka;
    uint32_t a_begin, a_count;      // tracks this launch works on
    uint32_t *error;
    uint32_t *has_long;             // out: set when an interval of >= 2^20 - 1 bases was filed
    unsigned long long *total;      // out: entries needed
};
size_t build_bins_scan_bytes(uint64_t n_boff);
cudaError_t launch_bins_count(cudaStream_t st, const BuildBinsParams &p);
cudaError_t launch_bins_finish(cudaStream_t st, const BuildBinsParams &p, void *scan_tmp, size_t scan_bytes);

// counter: GATB_* id.  Returns cudaError from the launch configuration.
cudaError_t launch_count(cudaStream_t st, int counter, const CountParams &p, int threads);

// diagnostic: segments and index entries in the runs of the placed segments (bench.py roofline)
void launch_count_work(cudaStream_t st, const CountParams &p, unsigned long long *out);

// column statistics (K5), column-tiled.  Pass 1 of a float64 matrix STORES sum, n_lt and n_eq; pass 1 of a uint32
// matrix ADDS its exact integers to isum, n_lt, n_eq, sq_lo and sq_hi (zeroed by the caller), so that successive slabs
// of rows give what one pass over all of them gives, and folds each column's extremes into col_min / col_max when
// col_min is set
struct StatsParams {
    const void *counts;             // [n_samples][n_cols] uint32 or float64
    int is_float;
    uint64_t n_samples;
    uint32_t n_cols;
    const double *observed;         // device [n_cols]; already divided by ref fold where applicable
    // outputs, device [n_cols]
    double *sum;                    // float64: sum (pass 1)
    double *sumsq_dev;              // float64: sum (x-mean)^2 (pass 2)
    unsigned long long *n_lt;       // #{ x < obs } = insertion point of obs (gat/Engine.pyx:1549-1557)
    unsigned long long *n_eq;       // #{ x == obs }
    unsigned long long *sq_lo, *sq_hi;   // uint32: exact sum of squares, 128 bits (the variance follows on the host)
    unsigned long long *isum;       // uint32: the exact integer sum
    double *q_lo, *q_hi;            // order statistics at ranks rank_lo / rank_hi (select)
    uint64_t rank_lo, rank_hi;
    const double *mean;             // float64: device [n_cols] (pass 2)
    uint64_t row_stride;            // pass 1: elements from one row to the next (0: n_cols)
    uint32_t *col_min, *col_max;    // uint32: per-column extremes, or NULL
};
// gat-compare (scripts/gat-compare.py:218-241, :300-323): the sampled log ratio of two fold-change columns,
//   out[s][p] = log((obs1[p] / (m1[s][col1[p]] + pc) + 1e-4) / (obs2[p] / (m2[s][col2[p]] + pc) + 1e-4)) + delta[p]
// for pairs p0 <= p < p0 + n_pairs; out is [n_samples][n_pairs] float64, ready for the column statistics
struct CompareParams {
    const double *m1, *m2;          // [n_samples][n_cols1], [n_samples][n_cols2]
    uint32_t n_cols1, n_cols2;
    uint64_t n_samples;
    const int32_t *col1, *col2;     // [n_pairs] (already offset to the chunk)
    const double *obs1, *obs2, *delta;
    uint32_t n_pairs;
    double pseudo_count;
    double *out;
};
void launch_compare_derive(cudaStream_t st, const CompareParams &p);

// counts table text (gat/__init__.py:1072-1086): column a of counts[n_samples][n_cols] as "c0,c1,...".
// Pass 1 (text == NULL): col_len[a] = bytes of column a.  Pass 2: the bytes, column a at text + col_off[a].
void launch_format_counts(cudaStream_t st, const uint32_t *counts, uint64_t n_samples, uint32_t n_cols,
                          unsigned long long *col_len, const unsigned long long *col_off, char *text);

// K5 as HBM-bound streaming passes over a uint32 matrix (stats_stream.cu): TMA bulk copies of whole rows into a
// shared-memory ring, thread = column
struct StreamStatsParams {
    const uint32_t *counts;         // [n_samples][n_cols], 16-byte aligned
    uint64_t n_samples;
    uint32_t n_cols;
    uint32_t rows_per_stage;        // rows of one ring stage (multiple of 4: every chunk starts 16-byte aligned)
    uint32_t n_chunks;              // chunks of rows_per_stage rows, dealt to the CTAs round-robin
    uint32_t n_stages, col_width;   // set by the launchers
    int use_tma;                    // 0: the matrix is not 16-byte aligned, the threads copy the chunks themselves
    // pass 1: the integers are ADDED to the caller's sums (ColumnSums in api.cu) with integer atomics
    // the comparison with the observed value as integer tests (set by stats_stream_thresholds):
    //   (double)v < observed  <=>  v < lt_thr  (or every v, flag 1);   (double)v == observed  <=>  flag 2 and v == eq_val
    const uint32_t *lt_thr, *eq_val, *col_flags;
    unsigned long long *isum, *n_lt, *n_eq;
    unsigned long long *sq_lo, *sq_hi;   // sum of squares, 128 bits
    uint32_t *vmax;                 // largest value of the matrix
    uint32_t *col_min, *col_max;    // extremes of every column folded in as well (MODE 2), or NULL (MODE 0)
    // select pass at bit `shift` (4 bits): prefix / rank per (which rank, column), [2][n_cols]
    uint32_t shift;
    uint32_t *prefix, *prefix_out;
    unsigned long long *rank, *rank_out;
    uint32_t *hist;                 // [2][16][n_cols], zero between passes
    double *q_lo, *q_hi;            // written by the last pass (shift 0)
    uint32_t *error;                // set when a TMA wait timed out
};
bool stats_stream_fits(const void *counts, uint64_t n_samples, uint32_t n_cols, size_t smem_optin);
void stats_stream_geometry(StreamStatsParams &p);
void stats_stream_thresholds(const double *observed, uint32_t n_cols, uint32_t *lt_thr, uint32_t *eq_val, uint32_t *flags);
cudaError_t launch_stats_stream_pass1(cudaStream_t st, StreamStatsParams p, int sm_count);
cudaError_t launch_stats_stream_select(cudaStream_t st, StreamStatsParams p, int sm_count, size_t smem_optin);

// Quantile-window histograms of a column accumulator (gatb_colacc_*).  Column a owns the unit-width uint32 bins
// [lo[a], lo[a] + width[a]) at bins + bin_off[a]; a value below / above its window counts into outside[a] /
// outside[n_cols + a].
struct ColHistParams {
    const uint32_t *counts;         // slab [n_rows][row_stride], the first n_cols of every row
    uint64_t n_rows, row_stride;
    uint32_t n_cols;
    const uint32_t *lo, *width;
    const unsigned long long *bin_off;
    uint32_t *bins;
    unsigned long long *outside;    // [2][n_cols]
    // pick: the values of ranks rank_lo / rank_hi of n_samples (the whole column: below + bins + above)
    uint64_t n_samples, rank_lo, rank_hi;
    uint32_t *q;                    // out [2][n_cols]
    unsigned long long *total;      // out [n_cols]: samples the histogram of the column holds
    uint32_t *missed;               // out [n_cols]: 1 when a rank falls below or above the window
};
cudaError_t launch_colacc_hist(cudaStream_t st, const ColHistParams &p, int sm_count);
cudaError_t launch_colacc_pick(cudaStream_t st, const ColHistParams &p);

void launch_stats_pass1(cudaStream_t st, const StatsParams &p);
void launch_stats_pass2(cudaStream_t st, const StatsParams &p);
void launch_stats_select(cudaStream_t st, const StatsParams &p);

}  // namespace gatb
