// stats_stream.cu -- K5 column statistics of a uint32 count matrix [sample][column] as HBM-bound streaming passes.  sm_100a.
//
// (gat/Engine.pyx:1635-1718 AnnotatorResult statistics, :1543-1576 getTwoSidedPValue.)  The matrix is S x A uint32,
// 4 GB at the north-star size, and every statistic is a per-column reduction over all rows: the passes are pure
// streaming and the roofline is the HBM copy bandwidth.  The column-tiled kernels of count.cu put only A / 16 CTAs
// on the machine (63 for 1000 columns, 8 for a column block of 125) and ran at a few percent of it.  Here a CTA owns
// whole ROWS: a chunk of `rows_per_stage` rows is one contiguous piece of memory, which the TMA unit copies into a
// ring of shared-memory stages (cp.async.bulk, completion on an mbarrier) while the threads -- thread = column,
// row lanes when there are fewer columns than threads -- work the previous stage off with conflict-free shared
// loads.  The grid is 2 CTAs per SM (1 for the select pass), chunks are dealt round-robin.
//   pass 1   sum x (uint64), sum x^2 (128 bits), #{x < observed}, #{x == observed}, max -- all integers, accumulated
//            with atomics: exact, so the results do not depend on the grid, the GPU or the column layout.  The
//            variance follows on the host from the exact n * sum x^2 - (sum x)^2 (no second pass over the matrix)
//            (pass 1 of a column accumulator, MODE 2: the same, plus the smallest and largest value of every column)
//   select   radix select of the two order statistics (CI bounds), 4 bits per pass from the highest non-zero
//            nibble of the matrix maximum: per-CTA histograms [rank][nibble][column] in shared memory, flushed to
//            global counters; stats_pick_kernel narrows prefix and rank between passes
#include <algorithm>
#include <cmath>

#include "count.cuh"
#include "ptx.cuh"

namespace gatb {

constexpr uint32_t SS_STAGE_BYTES = 32768;          // one stage of the ring
constexpr uint32_t SS_ALL_LESS = 1u, SS_HAS_EQUAL = 2u;   // StreamStatsParams.col_flags
constexpr uint32_t SS_WAIT_SPINS = 1u << 20;        // mbarrier polls before a CTA gives up (flags p.error: the call fails)

__host__ __device__ __forceinline__ uint32_t ss_hist_stride(uint32_t n_cols) { return ((n_cols + 31u) & ~31u) + 1u; }   // = 1 mod 32

// shared memory of a pass: [stages][mbarriers][select: histograms]
size_t stats_stream_smem(const StreamStatsParams &p, int mode, int threads)
{
    size_t b = (size_t)p.n_stages * SS_STAGE_BYTES + 64;
    if (mode == 1) b += (size_t)2 * 16 * ss_hist_stride(p.n_cols) * sizeof(uint32_t);
    (void)threads;
    return b;
}

// the CTA's j-th chunk is chunk blockIdx.x + j * gridDim.x of the matrix
struct ChunkSeq {
    uint32_t n_local;           // chunks of this CTA
    __device__ __forceinline__ uint64_t row0(const StreamStatsParams &p, uint32_t q) const
    {
        return ((uint64_t)blockIdx.x + (uint64_t)q * gridDim.x) * p.rows_per_stage;
    }
    __device__ __forceinline__ uint32_t rows(const StreamStatsParams &p, uint32_t q) const
    {
        return (uint32_t)min((uint64_t)p.rows_per_stage, p.n_samples - row0(p, q));
    }
};

// the bits above the nibble a select pass at `shift` decides
__host__ __device__ __forceinline__ uint32_t hmask_of(uint32_t shift) { return shift >= 28u ? 0u : (0xffffffffu << (shift + 4u)); }

// MODE 0: pass 1, 1: select pass, 2: pass 1 with per-column extremes.  KC = columns per thread (thread (c, r) owns columns c, c + CW, ...).  The inner
// loops address shared memory by 32-bit shared address and keep every per-element step to a handful of integer
// instructions (about 12 in pass 1, 8 in a select pass): at 4 bytes per element the passes only stay HBM-bound if
// the SMs can issue an element's work in the time its 4 bytes take to arrive.
template <int MODE, int KC>
__global__ void __launch_bounds__(1024) stats_stream_kernel(StreamStatsParams p)
{
    extern __shared__ __align__(16) uint8_t smem[];
    constexpr bool P1 = MODE != 1, MM = MODE == 2;
    const uint32_t T = blockDim.x, tid = threadIdx.x;
    const uint32_t CW = p.col_width, RW = T / CW;           // threads across columns, row lanes
    const uint32_t c = tid % CW, r = tid / CW;
    const uint32_t stage0 = smem_addr(smem);
    const uint32_t mbar0 = stage0 + p.n_stages * SS_STAGE_BYTES;
    const uint32_t hist0 = mbar0 + 64u;                     // MODE 1: [2][16][HS] counters
    const uint32_t row_bytes = p.n_cols * 4u;
    const uint32_t full_bytes = p.rows_per_stage * row_bytes;
    const uint32_t HS = ss_hist_stride(p.n_cols);

    ChunkSeq seq;
    seq.n_local = blockIdx.x < p.n_chunks ? (p.n_chunks - blockIdx.x + gridDim.x - 1u) / gridDim.x : 0u;
    const uint32_t n_chunks = seq.n_local;

    if (tid == 0) {
        for (uint32_t s = 0; s < p.n_stages; s++) mbar_init(mbar0 + 8u * s, 1u);
        fence_mbar_init();
    }
    if (MODE == 1)
        for (uint32_t i = tid; i < 2u * 16u * HS; i += T) sts32(hist0 + 4u * i, 0u);
    __syncthreads();

    // the TMA producer: one thread; a full chunk is ONE bulk copy (rows are contiguous), the partial chunk at the
    // very end of the matrix is copied by the threads themselves
    auto issue = [&](uint32_t q) {
        if (p.use_tma && q < n_chunks && seq.rows(p, q) == p.rows_per_stage) {
            const uint32_t s = q % p.n_stages;
            mbar_expect_tx(mbar0 + 8u * s, full_bytes);
            bulk_copy_g2s(stage0 + s * SS_STAGE_BYTES, p.counts + seq.row0(p, q) * p.n_cols, full_bytes, mbar0 + 8u * s);
        }
    };
    if (tid == 0)
        for (uint32_t q = 0; q < p.n_stages; q++) issue(q);

    // per-column state (a column past the end reads column 0 and is dropped when the results go out)
    bool live[KC];
    uint32_t coff[KC];                                      // byte offset of the column inside a row
    uint32_t neg_thr[KC], inv_eq[KC];                       // pass 1: 2^32 - lt_thr and ~eq_val (count_carry)
    unsigned long long sum[KC], sq_lo[KC];
    uint32_t sq_hi[KC], nge[KC], ngt[KC], vmax = 0, nrows = 0;
    uint32_t cmin[KC], cmax[KC];                            // MODE 2
    uint32_t pre0[KC], pre1[KC], h0[KC];                    // select: prefixes, shared address of the column's counters
#pragma unroll
    for (int k = 0; k < KC; k++) {
        const uint32_t col = c + (uint32_t)k * CW;
        live[k] = col < p.n_cols;
        coff[k] = live[k] ? col * 4u : 0u;
        neg_thr[k] = (P1 && live[k]) ? 0u - p.lt_thr[col] : 0u;
        inv_eq[k] = (P1 && live[k]) ? ~p.eq_val[col] : 0u;
        pre0[k] = (MODE == 1 && live[k]) ? p.prefix[col] : 0u;
        pre1[k] = (MODE == 1 && live[k]) ? p.prefix[p.n_cols + col] : 0u;
        // (a dead column counts into the padding slot HS - 1 of its rows, which is never flushed)
        h0[k] = pin_reg(hist0 + 4u * (live[k] ? col : HS - 1u));
        // while both ranks share their prefix one histogram serves both: the second comparison gets a value that
        // no masked element can take (bits outside the mask)
        if (MODE == 1 && pre0[k] == pre1[k]) pre1[k] = ~hmask_of(p.shift);
        pre0[k] = pin_reg(pre0[k]); pre1[k] = pin_reg(pre1[k]);
        coff[k] = pin_reg(coff[k]);
        sum[k] = sq_lo[k] = 0ull;
        sq_hi[k] = nge[k] = ngt[k] = 0u;
        cmin[k] = 0xffffffffu; cmax[k] = 0u;
    }
    const uint32_t hmask = pin_reg(hmask_of(p.shift));      // bits already decided
    const uint32_t HS4 = pin_reg(4u * HS), H1 = pin_reg(4u * 16u * HS), shift = pin_reg(p.shift);
    const uint32_t stage_base = pin_reg(stage0), rows_full = pin_reg(p.rows_per_stage);
    const uint32_t dummy = pin_reg(hist0 + 4u * (HS - 1u));  // (padding slot: never flushed)

    // (stage, parity and first row of the running chunk are carried along: no division per chunk)
    uint32_t s = 0, parity = 0;
    uint64_t row0 = (uint64_t)blockIdx.x * rows_full;
    const uint64_t row_step = (uint64_t)gridDim.x * rows_full;
    const uint32_t n_stages = pin_reg(p.n_stages);
    const bool use_tma = p.use_tma != 0;
    for (uint32_t q = 0; q < n_chunks; q++, row0 += row_step) {
        const uint32_t rows = row0 + rows_full <= p.n_samples ? rows_full : (uint32_t)(p.n_samples - row0);
        const uint32_t stage = stage_base + s * SS_STAGE_BYTES;
        int timed_out = 0;
        if (rows == rows_full && use_tma) {
            uint32_t spins = 0;
            while (!mbar_try_wait(mbar0 + 8u * s, parity))
                if (++spins > SS_WAIT_SPINS) { timed_out = 1; break; }
        } else if (rows) {                          // (the partial last chunk; every chunk of an unaligned matrix)
            const uint32_t *src = p.counts + row0 * p.n_cols;
            for (uint32_t i = tid; i < rows * p.n_cols; i += T) sts32(stage + 4u * i, src[i]);
            __syncthreads();
        }
#pragma unroll 4
        for (uint32_t row = r; row < rows; row += RW) {
            const uint32_t rowa = stage + row * row_bytes;
            if (P1) nrows++;
#pragma unroll
            for (int k = 0; k < KC; k++) {
                const uint32_t v = lds32(rowa + coff[k]);
                if (P1) {
                    sum[k] += v;
                    add96_sq(sq_lo[k], sq_hi[k], v);
                    count_carry(nge[k], v, neg_thr[k]);          // v >= lt_thr; searchargsorted + cmpDouble (gat/Engine.pyx:122-127, 1549-1557)
                    count_carry(ngt[k], v, inv_eq[k]);           // v > eq_val (#equal = #(>= t) - #(> t) when observed is an integer t)
                    vmax = max(vmax, v);
                    if (MM) { cmin[k] = min(cmin[k], v); cmax[k] = max(cmax[k], v); }
                } else {
                    // unconditional reductions (ptxas branches around a predicated one): an element that does not
                    // carry the prefix counts into a padding slot, where the hardware merges the lanes' increments
                    const uint32_t cell = ((v >> shift) & 15u) * HS4 + h0[k], hi = v & hmask;
                    red_add_shared(hi == pre0[k] ? cell : dummy, 1u);
                    red_add_shared(hi == pre1[k] ? cell + H1 : dummy, 1u);
                }
            }
        }
        // everyone is done with stage s: refill it.  (A copy that never completed -- it cannot, short of a broken
        // address -- ends the CTA's work for all of its threads at once and fails the call.)
        if (__syncthreads_or(timed_out)) {
            if (tid == 0) *p.error = 1u;
            break;
        }
        if (tid == 0) issue(q + n_stages);
        if (++s == n_stages) { s = 0; parity ^= 1u; }
    }

    if (P1) {
        // integers: exact and order-independent, one atomic per column, row lane and CTA.  The 128-bit sum of
        // squares: every atomic on the low word reports its own carry, whatever the order
#pragma unroll
        for (int k = 0; k < KC; k++) {
            const uint32_t col = c + (uint32_t)k * CW;
            if (live[k] && nrows) {
                const uint32_t fl = p.col_flags[col];
                const unsigned long long lo = sq_lo[k];
                unsigned long long hi = sq_hi[k];
                if (sum[k]) atomicAdd(p.isum + col, sum[k]);
                if (lo) {
                    const unsigned long long old = atomicAdd(p.sq_lo + col, lo);
                    hi += (old + lo < old) ? 1ull : 0ull;
                }
                if (hi) atomicAdd(p.sq_hi + col, hi);
                // lt_thr = 0: nothing is smaller (and the carry count is void: 2^32 - 0 wraps).  SS_HAS_EQUAL: observed is
                // an integer t and lt_thr = eq_val = t, so #equal = #(>= t) - #(> t); for t = 0 every row is >= t
                const uint32_t ge = p.lt_thr[col] ? nge[k] : nrows;
                const uint32_t lt = (fl & SS_ALL_LESS) ? nrows : nrows - ge, eq = (fl & SS_HAS_EQUAL) ? ge - ngt[k] : 0u;
                if (lt) atomicAdd(p.n_lt + col, (unsigned long long)lt);
                if (eq) atomicAdd(p.n_eq + col, (unsigned long long)eq);
                if (MM) { atomicMin(p.col_min + col, cmin[k]); atomicMax(p.col_max + col, cmax[k]); }
            }
        }
        vmax = __reduce_max_sync(GATB_FULL, vmax);
        if ((tid & 31u) == 0 && vmax) atomicMax(p.vmax, vmax);
    }
    if (MODE == 1) {
        __syncthreads();
        for (uint32_t i = tid; i < 2u * 16u * HS; i += T) {
            const uint32_t v = lds32(hist0 + 4u * i), col = i % HS;
            if (v && col < p.n_cols) atomicAdd(p.hist + (uint64_t)(i / HS) * p.n_cols + col, v);
        }
    }
}

// between two select passes: the nibble that holds the wanted rank extends the prefix; the histograms are cleared
__global__ void __launch_bounds__(256) stats_pick_kernel(StreamStatsParams p)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2u * p.n_cols) return;
    const uint32_t w = i / p.n_cols, col = i % p.n_cols;
    const bool shared_hist = p.prefix[col] == p.prefix[p.n_cols + col];      // (before either of them is updated)
    uint32_t *h = p.hist + (uint64_t)((w && !shared_hist) ? 16u : 0u) * p.n_cols + col;
    unsigned long long rank = p.rank[i], cum = 0;
    uint32_t b = 0;
    for (; b < 16u; b++) {
        const uint32_t v = h[(uint64_t)b * p.n_cols];
        if (cum + v > rank) break;
        cum += v;
    }
    if (b > 15u) b = 15u;
    // both ranks of a column may read the shared histogram: clear only after both have (second kernel phase below)
    p.rank_out[i] = rank - cum;
    p.prefix_out[i] = p.prefix[i] | (b << p.shift);
}
__global__ void __launch_bounds__(256) stats_pick_commit_kernel(StreamStatsParams p)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 2u * p.n_cols) {
        p.rank[i] = p.rank_out[i];
        p.prefix[i] = p.prefix_out[i];
        if (p.shift == 0) (i < p.n_cols ? p.q_lo : p.q_hi)[i % p.n_cols] = (double)p.prefix_out[i];
    }
    for (uint64_t j = i; j < 32ull * p.n_cols; j += (uint64_t)gridDim.x * blockDim.x) p.hist[j] = 0u;
}

template <int MODE>
static cudaError_t launch_stream_mode(cudaStream_t st, const StreamStatsParams &p, int sm_count)
{
    const int threads = MODE == 1 ? 1024 : 512;
    StreamStatsParams q = p;
    uint32_t cw = 1;
    while (cw < p.n_cols && cw < (uint32_t)threads) cw <<= 1;
    q.col_width = cw;
    const uint32_t kc = (p.n_cols + cw - 1u) / cw;
    const size_t smem = stats_stream_smem(q, MODE, threads);
    const unsigned grid = (unsigned)std::min<uint64_t>(p.n_chunks, (uint64_t)sm_count * (MODE == 1 ? 1u : 2u));
    cudaError_t e;
#define GATB_SS_LAUNCH(KC_)                                                                                                   \
    e = cudaFuncSetAttribute(stats_stream_kernel<MODE, KC_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);            \
    if (e != cudaSuccess) return e;                                                                                            \
    stats_stream_kernel<MODE, KC_><<<grid, threads, smem, st>>>(q);
    if (kc <= 1) { GATB_SS_LAUNCH(1) }
    else if (kc <= 2) { GATB_SS_LAUNCH(2) }
    else { GATB_SS_LAUNCH(4) }                      // (n_cols <= 2048, at least 512 threads)
#undef GATB_SS_LAUNCH
    return cudaGetLastError();
}

// can the streaming passes take this matrix?  (uint32, rows short enough for a stage, histograms that fit)
bool stats_stream_fits(const void *counts, uint64_t n_samples, uint32_t n_cols, size_t smem_optin)
{
    if (((uintptr_t)counts & 3u) != 0 || n_samples == 0 || n_samples >= (1ull << 32)) return false;
    if ((uint64_t)n_cols * 4u * 4u > SS_STAGE_BYTES) return false;                 // at least 4 rows per stage
    StreamStatsParams p;
    p.n_cols = n_cols; p.n_stages = 2;
    return stats_stream_smem(p, 1, 1024) <= smem_optin;
}

void stats_stream_geometry(StreamStatsParams &p)
{
    const uint32_t row_bytes = p.n_cols * 4u;
    p.rows_per_stage = std::max(4u, (SS_STAGE_BYTES / row_bytes) & ~3u);            // multiple of 4: chunks start 16-byte aligned
    p.n_chunks = (uint32_t)((p.n_samples + p.rows_per_stage - 1u) / p.rows_per_stage);
    // (a plane of a [counter][sample][column] tensor may start 4, 8 or 12 bytes off: same passes, the threads copy)
    p.use_tma = ((uintptr_t)p.counts & 15u) == 0 ? 1 : 0;
}

// the comparisons of pass 1 without floating point: for an integer v and a real t, v < t <=> v < ceil(t), and v == t
// only if t is itself an integer in range
void stats_stream_thresholds(const double *observed, uint32_t n_cols, uint32_t *lt_thr, uint32_t *eq_val, uint32_t *flags)
{
    for (uint32_t a = 0; a < n_cols; a++) {
        const double t = observed[a];
        lt_thr[a] = 0u; eq_val[a] = 0u; flags[a] = 0u;
        if (!(t > 0.0)) {                           // t <= 0 or NaN: nothing is smaller
            if (t == 0.0) flags[a] |= SS_HAS_EQUAL;
        } else if (t > 4294967295.0) flags[a] |= SS_ALL_LESS;
        else {
            const double up = ceil(t);
            lt_thr[a] = (uint32_t)up;
            if (up == t) { eq_val[a] = (uint32_t)t; flags[a] |= SS_HAS_EQUAL; }
        }
    }
}

cudaError_t launch_stats_stream_pass1(cudaStream_t st, StreamStatsParams p, int sm_count)
{
    p.n_stages = 3;
    return p.col_min ? launch_stream_mode<2>(st, p, sm_count) : launch_stream_mode<0>(st, p, sm_count);
}

// one 4-bit select pass at p.shift (prefix / rank / hist as the previous pass left them)
cudaError_t launch_stats_stream_select(cudaStream_t st, StreamStatsParams p, int sm_count, size_t smem_optin)
{
    // one CTA per SM (the histograms take most of its shared memory): as many stages as fit next to them, so that
    // more than one copy is in flight while a stage is being worked off
    p.n_stages = 4;
    while (p.n_stages > 2 && stats_stream_smem(p, 1, 1024) > smem_optin) p.n_stages--;
    cudaError_t e = launch_stream_mode<1>(st, p, sm_count);
    if (e != cudaSuccess) return e;
    const unsigned nb = (2u * p.n_cols + 255u) / 256u;
    stats_pick_kernel<<<nb, 256, 0, st>>>(p);
    stats_pick_commit_kernel<<<nb, 256, 0, st>>>(p);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------
// Quantile-window histograms (gatb_colacc_*): the two CI95 order statistics of a column without its samples.  Bins
// are exact values, so the ranks stay exact.  Thread = column of a row, CTAs stride over the rows: the 32 increments
// of a warp go to 32 different columns' windows, never to one address, and the arena (columns x window width x 4
// bytes) stays in L2, where the reductions (RED, no return value) are served.  Increments of the same bin from
// different rows are spread over time by the row stride of the grid.
constexpr uint32_t CH_THREADS = 256, CH_UNROLL = 4;

__global__ void __launch_bounds__(CH_THREADS) colacc_hist_kernel(ColHistParams p)
{
    const uint32_t a = blockIdx.x * CH_THREADS + threadIdx.x;
    if (a >= p.n_cols) return;
    const uint32_t lo = p.lo[a], w = p.width[a];
    uint32_t *bins = p.bins + p.bin_off[a];
    uint32_t below = 0, above = 0;
    const uint64_t step = gridDim.y;
    uint64_t row = blockIdx.y;
    for (; row + (CH_UNROLL - 1) * step < p.n_rows; row += CH_UNROLL * step) {
        uint32_t v[CH_UNROLL];
#pragma unroll
        for (uint32_t u = 0; u < CH_UNROLL; u++) v[u] = p.counts[(row + u * step) * p.row_stride + a];
#pragma unroll
        for (uint32_t u = 0; u < CH_UNROLL; u++) {
            const uint32_t d = v[u] - lo;               // (a value below the window wraps to >= w)
            if (d < w) atomicAdd(bins + d, 1u);
            else if (v[u] < lo) below++;
            else above++;
        }
    }
    for (; row < p.n_rows; row += step) {
        const uint32_t v = p.counts[row * p.row_stride + a], d = v - lo;
        if (d < w) atomicAdd(bins + d, 1u);
        else if (v < lo) below++;
        else above++;
    }
    if (below) atomicAdd(p.outside + a, (unsigned long long)below);
    if (above) atomicAdd(p.outside + p.n_cols + a, (unsigned long long)above);
}

// one CTA per column: the bins are cut into one run per thread, a scan of the run totals finds the run that holds
// each rank, and that thread walks its run to the bin
__global__ void __launch_bounds__(CH_THREADS) colacc_pick_kernel(ColHistParams p)
{
    __shared__ unsigned long long part[CH_THREADS + 1];
    const uint32_t a = blockIdx.x, tid = threadIdx.x;
    const uint32_t w = p.width[a];
    const uint32_t *bins = p.bins + p.bin_off[a];
    const unsigned long long below = p.outside[a], above = p.outside[p.n_cols + a];
    const uint32_t run = (w + CH_THREADS - 1u) / CH_THREADS;
    const uint32_t b0 = min(w, tid * run), b1 = min(w, b0 + run);
    unsigned long long s = 0;
    for (uint32_t b = b0; b < b1; b++) s += bins[b];
    part[tid + 1] = s;
    __syncthreads();
    if (tid == 0) {
        part[0] = below;
        for (uint32_t i = 1; i <= CH_THREADS; i++) part[i] += part[i - 1];     // part[i] = below + bins before run i
        const unsigned long long inside_end = part[CH_THREADS];
        p.total[a] = inside_end + above;
        const bool miss = p.rank_lo < below || p.rank_lo >= inside_end || p.rank_hi < below || p.rank_hi >= inside_end;
        p.missed[a] = miss ? 1u : 0u;
        if (miss) { p.q[a] = 0u; p.q[p.n_cols + a] = 0u; }
    }
    __syncthreads();
    const unsigned long long first = part[tid], last = part[tid + 1];
#pragma unroll
    for (int which = 0; which < 2; which++) {
        const unsigned long long rank = which ? p.rank_hi : p.rank_lo;
        if (rank < first || rank >= last) continue;
        unsigned long long cum = first;
        uint32_t b = b0;
        for (; b < b1; b++) {
            cum += bins[b];
            if (cum > rank) break;
        }
        p.q[(uint64_t)which * p.n_cols + a] = p.lo[a] + b;
    }
}

cudaError_t launch_colacc_hist(cudaStream_t st, const ColHistParams &p, int sm_count)
{
    if (p.n_rows == 0 || p.n_cols == 0) return cudaSuccess;
    const uint32_t gx = (p.n_cols + CH_THREADS - 1u) / CH_THREADS;
    // about 8 CTAs of 256 threads per SM, every CTA at least a few unrolled steps of rows
    const uint64_t gy = std::max<uint64_t>(1, std::min<uint64_t>((p.n_rows + 2 * CH_UNROLL - 1) / (2 * CH_UNROLL),
                                                                 std::max<uint64_t>(1, (uint64_t)sm_count * 8u / gx)));
    colacc_hist_kernel<<<dim3(gx, (unsigned)std::min<uint64_t>(gy, 65535u)), CH_THREADS, 0, st>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_colacc_pick(cudaStream_t st, const ColHistParams &p)
{
    if (p.n_cols == 0) return cudaSuccess;
    colacc_pick_kernel<<<p.n_cols, CH_THREADS, 0, st>>>(p);
    return cudaGetLastError();
}

}  // namespace gatb
