// common.cuh -- shared device helpers for the gat_b200 kernels (sm_100a).
//
// Segments are packed as uint64 = (start << 32) | end so that an unsigned 64-bit compare orders by
// start (then end), one 8-byte load fetches a segment, and a warp reads 32 segments as one 256-byte
// coalesced request.  All kernels are warp-synchronous: one warp owns one work unit.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#define GATB_FULL 0xffffffffu
#define GATB_KEY_INF 0xffffffffffffffffull

namespace gatb {

__host__ __device__ __forceinline__ uint64_t pack_seg(uint32_t s, uint32_t e) { return ((uint64_t)s << 32) | e; }
__host__ __device__ __forceinline__ uint32_t seg_start(uint64_t k) { return (uint32_t)(k >> 32); }
__host__ __device__ __forceinline__ uint32_t seg_end(uint64_t k) { return (uint32_t)k; }

__host__ __device__ __forceinline__ uint32_t next_pow2(uint32_t x)
{
    uint32_t p = 1;
    while (p < x) p <<= 1;
    return p;
}

// ---------------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11).  RNG contract (DESIGN.md): counter = (turn, block | track<<8,
// unit, sample), key = 64-bit seed.  Must stay bit-identical to oracle/gat_oracle.c:go_philox4x32_10.
struct Philox4 { uint32_t x, y, z, w; };

// The ten round keys of a seed, k[0][r] = k0 + r * 0x9E3779B9 and k[1][r] = k1 + r * 0xBB67AE85.  A kernel that takes
// them as a launch parameter reads them from the constant bank (into uniform registers, operands of the rounds' XORs)
// instead of rebuilding them at every inlined call.
struct PhiloxKeys { uint32_t k[2][10]; };

__host__ __device__ inline PhiloxKeys philox_keys(uint64_t seed)
{
    PhiloxKeys rk;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    for (int r = 0; r < 10; r++) {
        rk.k[0][r] = k0; rk.k[1][r] = k1;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return rk;
}

__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                          const PhiloxKeys &rk)
{
#pragma unroll
    for (int r = 0; r < 10; r++) {
#ifdef __CUDA_ARCH__
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
#else
        uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0, hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
#endif
        uint32_t n0 = hi1 ^ c1 ^ rk.k[0][r], n2 = hi0 ^ c3 ^ rk.k[1][r];
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    }
    Philox4 o; o.x = c0; o.y = c1; o.z = c2; o.w = c3;
    return o;
}

// floor(r64 * range / 2^64) for range < 2^32, r64 = rhi:rlo  -- unbiased to 2^-32 relative
__host__ __device__ __forceinline__ uint32_t bounded_u32(uint32_t rlo, uint32_t rhi, uint32_t range)
{
    return (uint32_t)(((uint64_t)rhi * range + (((uint64_t)rlo * range) >> 32)) >> 32);
}

#ifdef __CUDACC__
// ---------------------------------------------------------------------------------------------------
// warp primitives
__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

// A value that ptxas must keep in a register: it re-derives anything it can trace to a kernel parameter or a
// special register (LDC / S2R + arithmetic in every round of a hot loop) but not the result of a shuffle.
__device__ __forceinline__ uint32_t pin_reg(uint32_t v) { return __shfl_sync(GATB_FULL, v, (int)(threadIdx.x & 31u)); }

__device__ __forceinline__ int32_t warp_incl_scan_add(int32_t v)
{
    int lane = lane_id();
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int32_t t = __shfl_up_sync(GATB_FULL, v, d);
        if (lane >= d) v += t;
    }
    return v;
}

__device__ __forceinline__ uint32_t warp_incl_scan_add_u32(uint32_t v)
{
    int lane = lane_id();
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t t = __shfl_up_sync(GATB_FULL, v, d);
        if (lane >= d) v += t;
    }
    return v;
}

__device__ __forceinline__ int32_t warp_incl_scan_max(int32_t v)
{
    int lane = lane_id();
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int32_t t = __shfl_up_sync(GATB_FULL, v, d);
        if (lane >= d) v = max(v, t);
    }
    return v;
}

__device__ __forceinline__ uint64_t shfl_u64(uint64_t v, int src)
{
    uint32_t lo = __shfl_sync(GATB_FULL, (uint32_t)v, src);
    uint32_t hi = __shfl_sync(GATB_FULL, (uint32_t)(v >> 32), src);
    return ((uint64_t)hi << 32) | lo;
}

__device__ __forceinline__ uint64_t shfl_xor_u64(uint64_t v, int m)
{
    uint32_t lo = __shfl_xor_sync(GATB_FULL, (uint32_t)v, m);
    uint32_t hi = __shfl_xor_sync(GATB_FULL, (uint32_t)(v >> 32), m);
    return ((uint64_t)hi << 32) | lo;
}

// ---------------------------------------------------------------------------------------------------
// Warp bitonic sort of N = 2^k packed segments (ascending).  Strides >= 32 exchange through memory,
// strides < 32 run in registers with shuffles: the phases k = 2..32 take ONE load/store pass per
// 32-element block, every later phase one more.  The packed keys are a total order (start, then end),
// so both lanes of a compare-exchange agree on the outcome.
// Replaces SegmentList.sort() (gat/SegmentList.pyx:478-486, libc qsort by start).
__device__ __forceinline__ uint64_t cmpxchg_lane(uint64_t x, int lane, uint32_t jj, bool asc)
{
    const uint64_t y = shfl_xor_u64(x, (int)jj);
    const bool keep_min = (((lane & jj) == 0) == asc);
    return ((x > y) == keep_min) ? y : x;          // take the partner's key iff it is the one to keep
}

__device__ __forceinline__ void warp_bitonic_sort(uint64_t *buf, uint32_t N)
{
    const int lane = lane_id();
    if (N <= 1) return;
    // phases k = 2 .. min(N, 32): entirely inside aligned 32-element blocks
    for (uint32_t b0 = 0; b0 < N; b0 += 32) {
        const uint32_t i = b0 + lane;
        uint64_t x = (i < N) ? buf[i] : GATB_KEY_INF;   // N < 32: idle lanes carry +inf and never move below N
#pragma unroll
        for (uint32_t k = 2; k <= 32; k <<= 1) {
            if (k <= N) {
                const bool asc = ((i & k) == 0);
#pragma unroll
                for (uint32_t jj = 16; jj > 0; jj >>= 1)
                    if (jj < k) x = cmpxchg_lane(x, lane, jj, asc);
            }
        }
        if (i < N) buf[i] = x;
    }
    __syncwarp();
    for (uint32_t k = 64; k <= N; k <<= 1) {
        for (uint32_t j = k >> 1; j >= 32; j >>= 1) {
            for (uint32_t t = lane; t < (N >> 1); t += 32) {
                const uint32_t i = 2 * t - (t & (j - 1));
                const uint32_t p = i + j;
                const uint64_t a = buf[i], b = buf[p];
                const bool asc = ((i & k) == 0);
                if ((a > b) == asc) { buf[i] = b; buf[p] = a; }
            }
            __syncwarp();
        }
        for (uint32_t b0 = 0; b0 < N; b0 += 32) {       // strides 16 .. 1 in registers
            const uint32_t i = b0 + lane;
            uint64_t x = buf[i];
            const bool asc = ((i & k) == 0);
#pragma unroll
            for (uint32_t jj = 16; jj > 0; jj >>= 1) x = cmpxchg_lane(x, lane, jj, asc);
            buf[i] = x;
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------------
// Workspace of one unit: sorted disjoint pieces + inclusive cumulative lengths.
// Units with many pieces (isochore workspaces: ~160 tiles per unit) carry two BUCKET TABLES of WS_NB + 1 entries
// that narrow the binary searches below to the one or two pieces a bucket holds:
//   pick table  tab[b]             = first piece i with cuminc[i] > r_b, r_b = the smallest random base of bucket b
//   end table   tab[WS_NB + 1 + b] = first piece i with end[i] > x_b,    x_b = the smallest coordinate of bucket b
// bucket(v) = umulhi(v, inv) is monotone, so the answer for any value of bucket b lies in [tab[b], tab[b + 1]].
constexpr uint32_t WS_NB = 256;
struct WsView {
    const uint32_t *start;
    const uint32_t *end;
    const uint32_t *cuminc;   // cuminc[i] = sum_{j<=i} len_j   (SegmentListSampler.cdf + 1, gat/Engine.pyx:274-277)
    uint32_t n;
    const uint32_t *tabw;     // bucket tables, or nullptr: {pick_inv, end_inv, then 2 * (WS_NB + 1) 16-bit entries};
                              // bucket of a random base r = umulhi(r, pick_inv), of a coordinate x =
                              // umulhi(x - first workspace start, end_inv)
};
__device__ __forceinline__ const uint16_t *ws_tab16(const WsView &w) { return reinterpret_cast<const uint16_t *>(w.tabw + 2); }

// workspace bases in [0, x): prefix-coverage closed form (SURVEY App. A.2) -- replaces the two-pointer
// SegmentList.intersect + sum (gat/SegmentList.pyx:1469-1549, :1607-1616) used at every checkpoint.
__device__ __forceinline__ uint32_t ws_cov(const WsView &w, uint32_t x)
{
    if (w.n == 1) {
        uint32_t s = w.start[0], e = w.end[0];
        return x <= s ? 0u : (min(x, e) - s);
    }
    uint32_t lo = 0, hi = w.n;
    while (lo < hi) {                       // number of pieces with start < x
        uint32_t mid = (lo + hi) >> 1;
        if (w.start[mid] < x) lo = mid + 1; else hi = mid;
    }
    if (lo == 0) return 0u;
    uint32_t p = lo - 1;
    uint32_t before = p ? w.cuminc[p - 1] : 0u;
    return before + (min(x, w.end[p]) - w.start[p]);
}

// workspace bases in [s, e) = ws_cov(e) - ws_cov(s), with ONE search: the first piece ending after s, then the
// few pieces that start before e (segments are short against the pieces of an isochore workspace)
__device__ __forceinline__ uint32_t ws_overlap(const WsView &w, uint32_t s, uint32_t e)
{
    if (w.n == 1) return ws_cov(w, e) - ws_cov(w, s);
    if (e <= s) return 0u;
    uint32_t lo = 0, hi = w.n;
    if (w.tabw != nullptr) {
        const uint32_t first = w.start[0];
        const uint32_t b = s > first ? min(__umulhi(s - first, w.tabw[1]), WS_NB - 1u) : 0u;
        const uint16_t *t = ws_tab16(w);
        lo = t[WS_NB + 1u + b]; hi = t[WS_NB + 2u + b];
    }
    while (lo < hi) {                       // first piece with end > s
        const uint32_t mid = (lo + hi) >> 1;
        if (w.end[mid] > s) hi = mid; else lo = mid + 1;
    }
    uint32_t acc = 0;
    for (uint32_t p = lo; p < w.n; p++) {
        const uint32_t ps = w.start[p];
        if (ps >= e) break;
        acc += min(e, w.end[p]) - max(s, ps);
    }
    return acc;
}
// ---------------------------------------------------------------------------------------------------
// In-place merge(0) of a SORTED run of n packed segments (gat/SegmentList.pyx:756-816 with
// distance 0, after its sort): drop empty segments, join when start <= running max end (overlapping
// AND adjacent).  Returns the new count.  Warp-cooperative: prefix-max of ends across lanes, heads
// compacted with ballot/popc; the end of a merged segment is patched when the next head is met.
// With `ws` and `cov` the pass also returns the workspace coverage of the merged list
// (intersect(workspace).sum(), gat/Engine.pyx:593-599): element i adds the workspace bases of
// [max(start_i, running max end), end_i), the part of it that no earlier element covers.
// and `len` the total length of the merged list.
// NORMALIZE = true gives SegmentList.normalize instead (gat/SegmentList.pyx:697-754): only overlapping
// segments are joined, adjacent ones stay apart (`start >= max_end` opens a new segment).
template <bool NORMALIZE = false>
__device__ __forceinline__ uint32_t warp_merge0_sorted(uint64_t *buf, uint32_t n, const WsView *ws = nullptr,
                                                       uint32_t *cov = nullptr, uint32_t *len = nullptr)
{
    const int lane = lane_id();
    int32_t carry = -1;          // running max end of everything seen (int32 like the reference)
    uint32_t nout = 0, covered = 0, length = 0;
    // the element of the NEXT chunk is requested before this chunk's scan (the writes below stay behind the
    // chunk being read, so reading ahead is safe): the load latency hides behind the shuffles
    uint64_t ahead = ((uint32_t)lane < n) ? buf[lane] : 0;
    for (uint32_t b0 = 0; b0 < n; b0 += 32) {
        uint32_t i = b0 + lane;
        uint64_t x = ahead;
        ahead = (i + 32u < n) ? buf[i + 32u] : 0;
        int32_t s = (int32_t)seg_start(x), e = (int32_t)seg_end(x);
        bool valid = (i < n) && (s != e);
        int32_t ev = valid ? e : -1;
        int32_t incl = warp_incl_scan_max(ev);
        int32_t excl = __shfl_up_sync(GATB_FULL, incl, 1);
        if (lane == 0) excl = -1;
        int32_t prev_max = max(carry, excl);
        if (ws != nullptr && valid) {
            const int32_t lo = max(s, prev_max);
            if (e > lo) {
                covered += ws_overlap(*ws, (uint32_t)lo, (uint32_t)e);
                length += (uint32_t)(e - lo);
            }
        }
        bool head = valid && (NORMALIZE ? (s >= prev_max) : (s > prev_max));
        uint32_t hmask = __ballot_sync(GATB_FULL, head);
        uint32_t pos = nout + __popc(hmask & ((1u << lane) - 1));
        __syncwarp();                           // all lanes have read their element before any write
        if (head) {
            // high word = start of the new merged segment; low word (end) patched later
            reinterpret_cast<uint32_t *>(buf + pos)[1] = (uint32_t)s;
            if (pos > 0) reinterpret_cast<uint32_t *>(buf + pos - 1)[0] = (uint32_t)prev_max;
        }
        nout += __popc(hmask);
        carry = max(carry, __shfl_sync(GATB_FULL, incl, 31));
        __syncwarp();
    }
    if (nout > 0 && lane == 0) reinterpret_cast<uint32_t *>(buf + nout - 1)[0] = (uint32_t)carry;
    if (cov != nullptr) *cov = __reduce_add_sync(GATB_FULL, covered);
    if (len != nullptr) *len = __reduce_add_sync(GATB_FULL, length);
    __syncwarp();
    return nout;
}

// ---------------------------------------------------------------------------------------------------
// Counting sort for placements: their starts are spread evenly over the workspace, so bucketing by
// start (NB buckets over [min, max]) leaves about one key per bucket; a key's final position is its
// bucket's offset plus its rank among the bucket's few keys.  O(n) instead of the bitonic network's
// O(n log^2 n).  `tmp` = n free slots (not overlapping buf), `cnt` = GATB_SORT_NB words of this warp's
// shared memory.  Returns false, with buf untouched, when the keys are too clustered to gain anything
// (fragmented workspaces); the caller then runs the bitonic sort.  Equal keys are interchangeable, so
// the result is the same sequence either way.
constexpr uint32_t GATB_SORT_NB = 512;

// A plan = bucket range and count.  The caller may fix it beforehand (`plan`: lo <= every start, starts beyond
// the range share the last bucket) -- that saves the min / max pass over the keys -- and may even have
// counted the keys into `cnt` as it produced them (`prehist`), which saves the histogram pass as well.
struct SortPlan { uint32_t lo, inv, nb; };

__device__ __forceinline__ SortPlan make_sort_plan(uint32_t n, uint32_t lo, uint32_t hi)
{
    SortPlan pl;
    pl.lo = lo;
    pl.nb = min(GATB_SORT_NB, max(64u, next_pow2(n) >> 1));
    const uint64_t q = ((uint64_t)pl.nb << 32) / ((uint64_t)(hi - lo) + 1u);
    pl.inv = q > 0xffffffffull ? 0xffffffffu : (uint32_t)q;
    return pl;
}

__device__ __forceinline__ uint32_t sort_bucket(const SortPlan &pl, uint32_t start)
{
    return min(__umulhi(start - pl.lo, pl.inv), pl.nb - 1u);
}

__device__ __forceinline__ bool warp_bucket_sort(uint64_t *buf, uint32_t n, uint64_t *tmp, uint32_t *cnt,
                                                 const SortPlan *plan = nullptr, bool prehist = false)
{
    const int lane = lane_id();
    SortPlan pl;
    if (plan != nullptr) pl = *plan;
    else {
        uint32_t lo = 0xffffffffu, hi = 0u;
        for (uint32_t i = lane; i < n; i += 32) {
            const uint32_t s = seg_start(buf[i]);
            lo = min(lo, s); hi = max(hi, s);
        }
        lo = __reduce_min_sync(GATB_FULL, lo);
        hi = __reduce_max_sync(GATB_FULL, hi);
        pl = make_sort_plan(n, lo, hi);
    }
    const uint32_t NB = pl.nb;
    if (!prehist) {
        for (uint32_t b = lane; b < NB; b += 32) cnt[b] = 0u;
        __syncwarp();
        for (uint32_t i = lane; i < n; i += 32) atomicAdd(&cnt[sort_bucket(pl, seg_start(buf[i]))], 1u);
    }
    __syncwarp();
    uint32_t base = 0, mx = 0;                      // counts -> exclusive offsets, 32 buckets at a time
    for (uint32_t r = 0; r < NB; r += 32) {
        const uint32_t v = cnt[r + lane];
        mx = max(mx, v);
        const uint32_t incl = warp_incl_scan_add_u32(v);
        cnt[r + lane] = base + incl - v;
        base += __shfl_sync(GATB_FULL, incl, 31);
    }
    mx = __reduce_max_sync(GATB_FULL, mx);
    __syncwarp();
    if (mx > 64u && mx > 8u * (n / NB + 1u)) return false;
    for (uint32_t i = lane; i < n; i += 32) {
        const uint64_t key = buf[i];
        tmp[atomicAdd(&cnt[sort_bucket(pl, seg_start(key))], 1u)] = key;
    }
    __syncwarp();                                   // now cnt[b] = end of bucket b = start of bucket b + 1
    // rank inside the bucket; two keys per lane and pass, and four bucket mates of each per turn of the inner loop,
    // so that eight independent loads are in flight at once instead of two (a bucket holds a few keys, and each
    // turn waits for its loads)
    for (uint32_t j0 = lane; j0 < n; j0 += 64) {
        const uint32_t j1 = j0 + 32u;
        const bool has1 = j1 < n;
        const uint64_t key0 = tmp[j0], key1 = has1 ? tmp[j1] : 0ull;
        const uint32_t b0 = sort_bucket(pl, seg_start(key0)), b1 = has1 ? sort_bucket(pl, seg_start(key1)) : 0u;
        const uint32_t first0 = b0 ? cnt[b0 - 1u] : 0u, last0 = cnt[b0];
        const uint32_t first1 = has1 ? (b1 ? cnt[b1 - 1u] : 0u) : 0u, last1 = has1 ? cnt[b1] : 0u;
        const uint32_t m0 = last0 - first0, m1 = last1 - first1;
        uint32_t r0 = 0, r1 = 0;
        for (uint32_t t = 0; t < max(m0, m1); t += 4) {
            const uint32_t p0 = first0 + t, p1 = first1 + t;
            uint64_t x0[4], x1[4];      // (a slot past the bucket reads as +inf: never below a key, and past its own slot)
#pragma unroll
            for (uint32_t u = 0; u < 4; u++) {
                x0[u] = t + u < m0 ? tmp[p0 + u] : GATB_KEY_INF;
                x1[u] = t + u < m1 ? tmp[p1 + u] : GATB_KEY_INF;
            }
#pragma unroll
            for (uint32_t u = 0; u < 4; u++) {
                r0 += (x0[u] < key0 || (x0[u] == key0 && p0 + u < j0)) ? 1u : 0u;
                r1 += (x1[u] < key1 || (x1[u] == key1 && p1 + u < j1)) ? 1u : 0u;
            }
        }
        buf[first0 + r0] = key0;
        if (has1) buf[first1 + r1] = key1;
    }
    __syncwarp();
    return true;
}

// sort + merge(0) of n arbitrary packed segments in a buffer with at least next_pow2(n) slots; with
// `tmp` (n more free slots) and `cnt` given, mid-sized runs take the counting sort
template <bool NORMALIZE = false>
__device__ __forceinline__ uint32_t warp_sort_merge0(uint64_t *buf, uint32_t n, uint64_t *tmp = nullptr,
                                                     uint32_t *cnt = nullptr, const WsView *ws = nullptr,
                                                     uint32_t *cov = nullptr, uint32_t *len = nullptr,
                                                     const SortPlan *plan = nullptr, bool prehist = false)
{
    if (n == 0) { if (cov != nullptr) *cov = 0; if (len != nullptr) *len = 0; return 0; }
    const int lane = lane_id();
    if (tmp != nullptr && n >= 40u && n <= 32768u && warp_bucket_sort(buf, n, tmp, cnt, plan, prehist))
        return warp_merge0_sorted<NORMALIZE>(buf, n, ws, cov, len);
    uint32_t N = next_pow2(n);
    for (uint32_t i = n + lane; i < N; i += 32) buf[i] = GATB_KEY_INF;
    __syncwarp();
    warp_bitonic_sort(buf, N);
    return warp_merge0_sorted<NORMALIZE>(buf, n, ws, cov, len);
}

// merge(0) of a sorted, merged run U = buf[0,nu) with np <= 32 new segments stored behind it
// (buf[nu, nu+np)): the common checkpoint late in the placement loop, where one or two placements
// join an already merged list.  The new keys are sorted across lanes with shuffles, U is shifted
// right in place (top chunk first) by the number of new keys that precede each element, the new
// keys are dropped into the gaps and the usual merge(0) scan runs once.  O(nu/32) instead of a
// full bitonic sort.  Same result as warp_sort_merge0(buf, nu + np).
__device__ __forceinline__ uint32_t warp_insert_merge0(uint64_t *buf, uint32_t nu, uint32_t np,
                                                       const WsView *ws = nullptr, uint32_t *cov = nullptr,
                                                       uint32_t *len = nullptr)
{
    const int lane = lane_id();
    uint64_t key = ((uint32_t)lane < np) ? buf[nu + lane] : GATB_KEY_INF;
    // bitonic sort of the 32 lane-resident keys (ascending)
#pragma unroll
    for (uint32_t k = 2; k <= 32; k <<= 1) {
#pragma unroll
        for (uint32_t j = k >> 1; j > 0; j >>= 1) {
            key = cmpxchg_lane(key, lane, j, (lane & k) == 0);
        }
    }
    // insertion point of each new key in U: number of U elements <= key (ties keep U first)
    uint32_t pos = nu;
    if ((uint32_t)lane < np) {
        uint32_t lo = 0, hi = nu;
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (buf[mid] <= key) lo = mid + 1; else hi = mid;
        }
        pos = lo;
    }
    const uint32_t first = __shfl_sync(GATB_FULL, pos, 0);
    __syncwarp();
    // shift U[i] to i + #{new keys with pos <= i}, chunks from the top down so nothing unread is overwritten
    if (nu > first) {
        const uint32_t lowest_chunk = first >> 5;
        for (int c = (int)((nu - 1) >> 5); c >= (int)lowest_chunk; c--) {
            const uint32_t i = ((uint32_t)c << 5) + lane;
            const uint64_t x = (i < nu) ? buf[i] : 0;
            uint32_t cnt = 0;                      // upper_bound of i in the lane-resident sorted pos[]
#pragma unroll
            for (int step = 16; step > 0; step >>= 1) {
                const uint32_t probe = __shfl_sync(GATB_FULL, pos, (int)(cnt + step - 1));
                if (cnt + step <= np && probe <= i) cnt += step;
            }
            __syncwarp();
            if (i < nu && i >= first) buf[i + cnt] = x;
            __syncwarp();
        }
    }
    if ((uint32_t)lane < np) buf[pos + lane] = key;
    __syncwarp();
    return warp_merge0_sorted(buf, nu + np, ws, cov, len);
}

#endif  // __CUDACC__

}  // namespace gatb
