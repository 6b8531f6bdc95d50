// count.cu -- K3/K4 counting kernel, construction of the annotation grid index, and K5 column statistics.  sm_100a.
//
// Counting: a CTA owns (group of tracks -- normally ALL tracks) x (chunk of samples) and keeps the chunk's
// count matrix [sample][track] in shared memory.  It walks the keys (contigs) in order; the work of a key is
// cut into ITEMS of 32 consecutive segments of one sample (lane = segment), handed to the warps through a
// shared-memory counter, so that no warp waits for another.  A lane turns its segment into the TWO runs of
// grid-index entries that can overlap it (count.cuh: intervals open at the left edge of its first bin, and
// intervals starting in its bins; four 4-byte offset loads); the warp then works the up to 64 runs off as ONE flat
// sequence of entry PAIRS (lists hold an even number of entries), 32 pairs per round with every lane busy:
// which run a flat position belongs to comes from a warp OR-reduction (redux.sync) of the runs' first
// positions, the run's segment from a 16-byte shared-memory load.  Per pair: one 16-byte load; per
// entry the overlap test and an integer atomic into the (sample, track) accumulator.  Three items are in
// flight per warp -- segment load / bin-offset loads / entry rounds -- and the rounds themselves run as a
// branch-free three-stage pipeline (ownership, entry loads, counting), which hides the L2, shared-memory and
// REDUX latencies of this gather-bound kernel.  The index of one key (a few tens of MB at 1000 tracks) stays in L2 while the CTAs
// walk the keys in the same order.  The float64 nucleotide-density sum is formed per key from the integers,
// in the same key order and with the same compensated summation as the reference's Python sum()
// (gat/__init__.py:583-587).
#include <algorithm>
#include <cub/device/device_scan.cuh>
#include <cub/block/block_scan.cuh>
#include "count.cuh"
#include "ptx.cuh"
#include "../../include/gat_b200.h"

namespace gatb {

constexpr uint32_t NO_ITEM = 0xffffffffu;

// shared memory: per-warp staging (64 runs x (16 B segment + 4 B previous end)), accumulators, item tables
__host__ __device__ __forceinline__ size_t count_smem_fixed(uint32_t nwarps) { return (size_t)nwarps * 64u * 20u; }

size_t count_smem_bytes(uint32_t schunk, uint32_t ka, uint32_t kgrp, int threads, bool density)
{
    return count_smem_fixed((uint32_t)threads / 32u) + (size_t)schunk * ka * (density ? 20u : 4u) +
           (size_t)kgrp * (2u * schunk + 2u) * 4u + 16u;
}

template <int COUNTER> struct NeedPrevInterval { static constexpr bool value = COUNTER == GATB_SEGMENT_OVERLAP || COUNTER == GATB_SEGMENT_MIDOVERLAP; };
template <int COUNTER> struct NeedPrevSegment { static constexpr bool value = COUNTER == GATB_ANNOTATION_OVERLAP || COUNTER == GATB_ANNOTATION_MIDOVERLAP; };

// one PAIR of adjacent entries of the flat sequence, loaded two rounds ahead of its use
struct Flight {
    uint4 w;            // the two packed entries (one 16-byte load: runs start and end on even indices)
    uint32_t owner;     // staging slot of their segment
    uint32_t j;         // index of the first of the two
    uint2 pv;           // ends of the previous intervals of their tracks (segment-* counters)
};

// ---------------------------------------------------------------------------------------------------
// One live entry against its segment [s,e).  Every overlapping (segment, interval) pair is met exactly once
// (count.cuh), so the overlap test is all there is.  Coordinates are < 2^31.
//   nucleotide-overlap   overlapWithSegments            gat/SegmentList.pyx:1026-1076
//   segment-overlap      intersectionWithSegments(base) :1078-1146  (a segment counts once per track:
//                        at the first interval of the track that overlaps it, i.e. previous end <= s)
//   segment-midoverlap   midpoint tested against that FIRST overlapping interval only (:1137-1144)
//   annotation-*         roles swapped: an interval is counted by the first segment overlapping it,
//                        i.e. when it does not already overlap the previous segment (x >= pe)
//   overlap-pieces       len(a.intersect(b)): every overlapping pair is one piece (:1469-1549)
template <int COUNTER>
__device__ __forceinline__ void count_entry(uint32_t x, uint32_t wy, uint32_t y, uint32_t pv,
                                            const uint4 o, uint32_t pe, uint32_t acc_addr)
{
    const uint32_t s = o.x, e = o.y;                        // the entry's segment
    if (!((x < e) & (y > s))) return;
    const uint32_t cell = acc_cell(wy, acc_addr);
    if (COUNTER == GATB_NUCLEOTIDE_OVERLAP) {
        red_add_shared(cell, min(e, y) - max(s, x));
    } else if (COUNTER == GATB_SEGMENT_OVERLAP) {
        if (pv <= s) red_add_shared(cell, 1u);
    } else if (COUNTER == GATB_SEGMENT_MIDOVERLAP) {
        const uint32_t mid = s + ((e - s) >> 1);
        if (pv <= s && x <= mid && mid < y) red_add_shared(cell, 1u);
    } else if (COUNTER == GATB_OVERLAP_PIECES) {
        red_add_shared(cell, 1u);
    } else if (COUNTER == GATB_ANNOTATION_OVERLAP) {
        if (x >= pe) red_add_shared(cell, 1u);
    } else {
        const uint32_t m = x + ((y - x) >> 1);
        if (x >= pe && s <= m && m < e) red_add_shared(cell, 1u);
    }
}

// the two entries of a flight against their segment
template <int COUNTER, bool LONG>
__device__ __forceinline__ void count_pair(const uint2 *__restrict__ civ, const Flight &f, uint32_t stg, uint32_t stg_pe,
                                           uint32_t acc_addr)
{
    // (the segment is the first 8 bytes of the run's staging slot: an 8-byte shared load is 2 data-pipe wavefronts
    // for a warp, a 16-byte one 4 -- and that pipe is what the kernel saturates)
    const uint2 so = lds64(stg + f.owner * 16u);
    const uint4 o = make_uint4(so.x, so.y, 0u, 0u);
    uint32_t pe = 0;
    if (NeedPrevSegment<COUNTER>::value) pe = lds32(stg_pe + f.owner * 4u);
    // end = start + length; a length field of 2^20 - 1 sends us to civ[] for the end.  LONG = false: the index
    // holds no such interval (known after the build), and the kernel is compiled without the test
    uint32_t y0 = f.w.x + (f.w.y >> 12), y1 = f.w.z + (f.w.w >> 12);
    if (LONG) {
        if ((f.w.y >> 12) == ENTRY_LEN_MASK) y0 = civ[f.j].y;
        if ((f.w.w >> 12) == ENTRY_LEN_MASK) y1 = civ[f.j + 1u].y;
    }
    count_entry<COUNTER>(f.w.x, f.w.y, y0, f.pv.x, o, pe, acc_addr);
    count_entry<COUNTER>(f.w.z, f.w.w, y1, f.pv.y, o, pe, acc_addr);
}

// an item whose bin offsets have been requested: lane = segment
struct Indexed {
    uint32_t slot;              // sample slot in the chunk, NO_ITEM: none
    uint32_t s, e, pe;
    uint32_t c0, c1;            // C[b0]: intervals open at the left edge of the segment's first bin
    uint32_t s0, s1;            // S[b0..b1]: intervals starting in the segment's bins
};

// The 32 runs [r0, r1) of an item as one flat sequence of entries.  stg / stg_pe: shared addresses of the
// warp's staging, acc_addr: of the sample's accumulators.
struct WarpConsts {
    uint32_t lane, le_mask, stg, stg_pe, sentinel;
    uint64_t cent;                                  // global address of the entry array
};

template <int COUNTER, bool LONG>
__device__ __forceinline__ void run_item(const CountParams &p, const WarpConsts &wc, const Indexed &it, uint32_t acc_addr)
{
    const uint32_t lane = wc.lane, stg = wc.stg, stg_pe = wc.stg_pe;
    // every list holds an even number of entries (padded with an entry that overlaps nothing) and starts on an
    // even index, so runs are whole PAIRS of entries: a lane takes a pair per round with one 16-byte load.
    // Flat order: lane 0's C run, lane 0's S run, lane 1's C run, ...
    const uint32_t len_c = (it.c1 - it.c0) >> 1, len_s = (it.s1 - it.s0) >> 1;      // pairs
    const uint32_t len = len_c + len_s;
    const uint32_t incl = warp_incl_scan_add_u32(len);
    const uint32_t total = __shfl_sync(GATB_FULL, incl, 31);
    if (total == 0) return;
    const uint32_t excl = incl - len;
    const uint32_t lt_mask = wc.le_mask >> 1;
    const uint32_t rank_c = __popc(__ballot_sync(GATB_FULL, len_c != 0u) & lt_mask) +
                            __popc(__ballot_sync(GATB_FULL, len_s != 0u) & lt_mask);
    const uint32_t rank_s = rank_c + (len_c != 0u ? 1u : 0u);
    __syncwarp();                                   // the previous item's readers are done with the staging
    if (len_c) {
        sts128(stg + rank_c * 16u, make_uint4(it.s, it.e, it.c0 - 2u * excl, 0u));
        if (NeedPrevSegment<COUNTER>::value) sts32(stg_pe + rank_c * 4u, it.pe);
    }
    if (len_s) {
        sts128(stg + rank_s * 16u, make_uint4(it.s, it.e, it.s0 - 2u * (excl + len_c), 0u));
        if (NeedPrevSegment<COUNTER>::value) sts32(stg_pe + rank_s * 4u, it.pe);
    }
    __syncwarp();
    const uint64_t cent = wc.cent;
    const uint32_t *__restrict__ cprev = p.cprev;
    const uint32_t le_mask = wc.le_mask, sentinel = wc.sentinel;
    // flat pair positions of the lane's two runs' first pairs (none: never matches a round)
    const uint32_t first_c = len_c ? excl : 0xffffffffu, first_s = len_s ? excl + len_c : 0xffffffffu;
    uint32_t started = 0xffffffffu;                 // (non-empty runs that begin before the round) - 1

    // Rounds of 32 flat pair positions, software-pipelined without branches: stage A (who owns the positions of
    // a round: one warp OR-reduction) runs three rounds ahead of the round being counted, stage B (the entry
    // loads) two rounds ahead.  Rounds past the end are harmless: no run starts there (owner = the last run)
    // and their positions are >= total (the sentinel pair).
    auto stage_a = [&](uint32_t base) -> uint32_t {
        const uint32_t mask = __reduce_or_sync(GATB_FULL, shl_clamp(1u, first_c - base) | shl_clamp(1u, first_s - base));
        const uint32_t owner = started + __popc(mask & le_mask);
        started += __popc(mask);
        return owner;
    };
    auto stage_b = [&](uint32_t base, Flight &f) {
        const uint32_t pos = base + lane;
        const uint32_t z = lds32(stg + f.owner * 16u + 8u);         // (first entry of the run) - 2 * (its flat pair position)
        f.j = (pos < total) ? 2u * pos + z : sentinel;
        f.w = ldg_nc_u4(cent + (uint64_t)f.j * 8u);
        if (NeedPrevInterval<COUNTER>::value) f.pv = *reinterpret_cast<const uint2 *>(cprev + f.j);
    };
    Flight f0, f1, f2;
    f0.owner = stage_a(0u); f1.owner = stage_a(32u); f2.owner = stage_a(64u);
    stage_b(0u, f0);
    stage_b(32u, f1);
    for (uint32_t base = 0;;) {
        stage_b(base + 64u, f2);
        count_pair<COUNTER, LONG>(p.civ, f0, stg, stg_pe, acc_addr);
        f0.owner = stage_a(base + 96u);
        base += 32u;
        if (base >= total) break;
        stage_b(base + 64u, f0);
        count_pair<COUNTER, LONG>(p.civ, f1, stg, stg_pe, acc_addr);
        f1.owner = stage_a(base + 96u);
        base += 32u;
        if (base >= total) break;
        stage_b(base + 64u, f1);
        count_pair<COUNTER, LONG>(p.civ, f2, stg, stg_pe, acc_addr);
        f2.owner = stage_a(base + 96u);
        base += 32u;
        if (base >= total) break;
    }
}

template <int COUNTER, bool DENSITY, bool LONG>
__global__ void __launch_bounds__(1024, 1) count_kernel(CountParams p)
{
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t lane = pin_reg(threadIdx.x & 31u);
    const int warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const uint32_t g = blockIdx.x;
    const uint32_t a0 = g * p.ka;
    const uint32_t ka = min(p.ka, p.n_annot - a0);
    const uint32_t s_begin = blockIdx.y * p.schunk;
    const uint32_t s_end = min(s_begin + p.schunk, p.n_samples);
    const uint32_t ns = s_end - s_begin, ncells = ns * ka;
    // layout: [staging][density only: (sum, compensation) doubles per cell][u32 per cell][item tables]
    WarpConsts wc;
    wc.lane = lane;
    wc.le_mask = pin_reg(0xffffffffu >> (31u - lane));
    wc.stg = pin_reg(smem_addr(smem) + (uint32_t)warp * 1024u);
    wc.stg_pe = pin_reg(smem_addr(smem) + (uint32_t)nwarps * 1024u + (uint32_t)warp * 256u);
    wc.sentinel = pin_reg(p.sentinel);
    {
        const uint64_t c = (uint64_t)__cvta_generic_to_global(p.cent);
        wc.cent = ((uint64_t)pin_reg((uint32_t)(c >> 32)) << 32) | pin_reg((uint32_t)c);
    }
    uint8_t *base = smem + count_smem_fixed((uint32_t)nwarps);
    double *acc_d = reinterpret_cast<double *>(base);
    uint32_t *acc_u = reinterpret_cast<uint32_t *>(base + (DENSITY ? (size_t)p.schunk * p.ka * 16u : 0u));
    // per key of the current key group: pre[slot] = items before sample slot (ns + 1), nn[slot] = its
    // number of segments on the key, cnt = next item to hand out
    uint32_t *pre = acc_u + (size_t)p.schunk * p.ka;
    uint32_t *nn = pre + (size_t)p.kgrp * (p.schunk + 1u);
    uint32_t *cnt = nn + (size_t)p.kgrp * p.schunk;
    const uint32_t acc_base = pin_reg(smem_addr(acc_u));

    for (uint32_t i = threadIdx.x; i < ncells; i += blockDim.x) {
        acc_u[i] = 0u;
        if (DENSITY) { acc_d[2 * i] = 0.0; acc_d[2 * i + 1] = 0.0; }
    }

    for (uint32_t k0 = 0; k0 < p.n_keys; k0 += p.kgrp) {
        const uint32_t nk = min(p.kgrp, p.n_keys - k0);
        __syncthreads();                                   // everyone is done with the previous tables
        for (uint32_t kk = (uint32_t)warp; kk < nk; kk += (uint32_t)nwarps) {
            const uint32_t k = k0 + kk;
            const KeyBins kb = p.keybins[(uint64_t)g * p.n_keys + k];
            // no interval of any track on this key / density: counter returns 0 (gat/Engine.pyx:1438-1440)
            const bool dead = kb.nbins == 0 || (DENSITY && p.key_ws_nseg[k] == 0);
            uint32_t run = 0;
            for (uint32_t q0 = 0; q0 < ns; q0 += 32) {
                const uint32_t slot = q0 + lane;
                uint32_t n = 0;
                if (slot < ns && !dead) {
                    const uint64_t sl = s_begin + slot;
                    if (!p.key_present || p.key_present[sl * p.n_keys + k]) n = p.placed_n[sl * p.n_keys + k];
                }
                const uint32_t incl = warp_incl_scan_add_u32((n + 31u) >> 5);
                if (slot < ns) {
                    nn[kk * p.schunk + slot] = n;
                    pre[kk * (p.schunk + 1u) + slot + 1u] = run + incl;
                }
                run += __shfl_sync(GATB_FULL, incl, 31);
            }
            if (lane == 0) { pre[kk * (p.schunk + 1u)] = 0u; cnt[kk] = 0u; }
        }
        __syncthreads();

        for (uint32_t kk = 0; kk < nk; kk++) {
            const uint32_t k = k0 + kk;
            const uint32_t *pre_k = pre + kk * (p.schunk + 1u);
            const uint32_t *nn_k = nn + kk * p.schunk;
            const uint32_t n_items = pre_k[ns];
            if (n_items) {
                const KeyBins kb = p.keybins[(uint64_t)g * p.n_keys + k];
                const uint4 *__restrict__ brec = p.brec + kb.base;
                const uint32_t *__restrict__ soff = p.boff + kb.base;
                const uint32_t *__restrict__ coff = p.boff + p.coff_base + kb.base;
                const uint64_t *__restrict__ placed_key = p.placed + p.key_base[k] + (uint64_t)s_begin * p.sample_stride;
                // three items in flight: A = segment requested, B = bin offsets requested, then run
                uint32_t a_slot = NO_ITEM, a_i = 0, a_n = 0, a_prev = 0;
                uint64_t a_sg = 0;
                Indexed b;
                b.slot = NO_ITEM;
                bool more = true;
                uint32_t cursor = 0;
                while (more || a_slot != NO_ITEM || b.slot != NO_ITEM) {
                    // A -> B': the segment has arrived; request its bin offsets
                    Indexed nb;
                    nb.slot = a_slot;
                    nb.s = nb.e = nb.pe = nb.c0 = nb.c1 = nb.s0 = nb.s1 = 0u;
                    if (a_slot != NO_ITEM) {
                        if (a_i < a_n) {
                            nb.s = seg_start(a_sg); nb.e = seg_end(a_sg);
                            const uint32_t b0 = nb.s >> kb.shift;
                            if (b0 < kb.nbins) {
                                const uint32_t b1 = min((nb.e - 1u) >> kb.shift, kb.nbins - 1u);
                                // ONE 16-byte record per segment (count.cuh): 32 lanes = 32 scattered sectors per
                                // load, so the NUMBER of loads per item is what the L1 data pipe pays for.  A
                                // segment reaching beyond b0 + 2, or a list too long for the 16-bit fields, reads
                                // the plain offset arrays instead (few lanes, rarely)
                                const uint4 r0 = brec[b0];
                                const uint32_t d = b1 - b0;
                                const uint32_t len_c = r0.z & 0xffffu;
                                const uint32_t len_s = d == 0u ? (r0.z >> 16) : d == 1u ? (r0.w & 0xffffu) : (r0.w >> 16);
                                nb.c0 = r0.x; nb.c1 = r0.x + len_c; nb.s0 = r0.y; nb.s1 = r0.y + len_s;
                                if (d > 2u || len_c == 0xffffu || len_s == 0xffffu) {
                                    nb.c1 = coff[b0 + 1u];
                                    nb.s1 = soff[b1 + 1u];
                                }
                            }
                        }
                        if (NeedPrevSegment<COUNTER>::value) {
                            nb.pe = __shfl_up_sync(GATB_FULL, nb.e, 1);
                            if (lane == 0) nb.pe = a_prev;
                        }
                    }
                    // next A: take an item, request its segments
                    a_slot = NO_ITEM;
                    if (more) {
                        uint32_t w = 0;
                        if (lane == 0) w = atomicAdd(cnt + kk, 1u);
                        w = __shfl_sync(GATB_FULL, w, 0);
                        if (w >= n_items) more = false;
                        else {
                            while (true) {                  // items come in increasing order: scan forward
                                const uint32_t idx = cursor + lane;
                                const uint32_t m = __ballot_sync(GATB_FULL, idx >= ns || pre_k[idx + 1u] > w);
                                if (m) { cursor += (uint32_t)__ffs(m) - 1u; break; }
                                cursor += 32u;
                            }
                            a_slot = cursor;
                            a_n = nn_k[cursor];
                            a_i = (w - pre_k[cursor]) * 32u + lane;
                            const uint64_t *segs = placed_key + (uint64_t)cursor * p.sample_stride;
                            if (a_i < a_n) a_sg = segs[a_i];
                            if (NeedPrevSegment<COUNTER>::value)
                                a_prev = (lane == 0 && a_i > 0u && a_i < a_n) ? seg_end(segs[a_i - 1u]) : 0u;
                        }
                    }
                    // run B (its offsets were requested one turn ago), then B <- B'
                    if (b.slot != NO_ITEM) run_item<COUNTER, LONG>(p, wc, b, acc_base + b.slot * ka * 4u);
                    b = nb;
                }
            }
            if (DENSITY) {
                // per key: float(overlap) / len(workspace), accumulated in key order like the reference's
                // Python sum(): CPython >= 3.12 sums floats with Neumaier compensation (Python/bltinmodule.c)
                __syncthreads();
                const uint32_t nseg = p.key_ws_nseg[k];
                if (n_items && nseg) {
                    const double den = (double)nseg;
                    for (uint32_t i = threadIdx.x; i < ncells; i += blockDim.x) {
                        const uint32_t v = acc_u[i];
                        if (v) {
                            const double x = (double)v / den, f = acc_d[2 * i], t = f + x;
                            acc_d[2 * i + 1] += (fabs(f) >= fabs(x)) ? ((f - t) + x) : ((x - t) + f);
                            acc_d[2 * i] = t;
                            acc_u[i] = 0u;
                        }
                    }
                }
                __syncthreads();
            }
        }
    }
    __syncthreads();
    if (!DENSITY && p.n_routes) {
        // routed delivery (count.cuh OutRoute): the finished rows go straight to their consumers, local or on a
        // peer GPU; consecutive threads write consecutive columns of one row (coalesced 4-byte stores)
        for (uint32_t i = threadIdx.x; i < ncells; i += blockDim.x) {
            const uint32_t row = s_begin + i / ka, a = a0 + i % ka, v = acc_u[i];
            for (uint32_t r = 0; r < p.n_routes; r++) {
                const OutRoute &rt = p.routes[r];
                if (a >= rt.col_begin && a < rt.col_end) rt.base[(rt.row0 + row) * rt.row_stride + (a - rt.col_begin)] = v;
            }
        }
        return;
    }
    for (uint32_t i = threadIdx.x; i < ncells; i += blockDim.x) {
        const uint64_t o = (uint64_t)(s_begin + i / ka) * p.n_annot + a0 + i % ka;
        if (DENSITY) {
            const double f = acc_d[2 * i], c = acc_d[2 * i + 1];
            p.out_f64[o] = (c != 0.0 && isfinite(c)) ? f + c : f;
        } else p.out_u32[o] = acc_u[i];
    }
}

template <int COUNTER, bool DENSITY, bool LONG>
static cudaError_t launch_count_tl(cudaStream_t st, const CountParams &p, int threads)
{
    const size_t smem = count_smem_bytes(p.schunk, p.ka, p.kgrp, threads, DENSITY);
    cudaError_t e = cudaFuncSetAttribute(count_kernel<COUNTER, DENSITY, LONG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    dim3 grid(p.n_groups, (p.n_samples + p.schunk - 1) / p.schunk);
    count_kernel<COUNTER, DENSITY, LONG><<<grid, threads, smem, st>>>(p);
    return cudaGetLastError();
}

template <int COUNTER, bool DENSITY>
static cudaError_t launch_count_t(cudaStream_t st, const CountParams &p, int threads)
{
    return p.has_long ? launch_count_tl<COUNTER, DENSITY, true>(st, p, threads) : launch_count_tl<COUNTER, DENSITY, false>(st, p, threads);
}

cudaError_t launch_count(cudaStream_t st, int counter, const CountParams &p, int threads)
{
    if (p.n_samples == 0 || p.n_annot == 0) return cudaSuccess;
    switch (counter) {
    case GATB_NUCLEOTIDE_OVERLAP:    return launch_count_t<GATB_NUCLEOTIDE_OVERLAP, false>(st, p, threads);
    case GATB_NUCLEOTIDE_DENSITY:    return launch_count_t<GATB_NUCLEOTIDE_OVERLAP, true>(st, p, threads);
    case GATB_SEGMENT_OVERLAP:       return launch_count_t<GATB_SEGMENT_OVERLAP, false>(st, p, threads);
    case GATB_SEGMENT_MIDOVERLAP:    return launch_count_t<GATB_SEGMENT_MIDOVERLAP, false>(st, p, threads);
    case GATB_ANNOTATION_OVERLAP:    return launch_count_t<GATB_ANNOTATION_OVERLAP, false>(st, p, threads);
    case GATB_ANNOTATION_MIDOVERLAP: return launch_count_t<GATB_ANNOTATION_MIDOVERLAP, false>(st, p, threads);
    case GATB_OVERLAP_PIECES:        return launch_count_t<GATB_OVERLAP_PIECES, false>(st, p, threads);
    }
    return cudaErrorInvalidValue;
}

// Diagnostic for bench.py's roofline: how many index entries the counting kernel has to test for the placed
// segments of a batch (the lengths of their runs, padding included) -- next to the number of truly overlapping
// pairs (the GATB_OVERLAP_PIECES counter) this is the kernel's waste ratio.  out[0] += segments, out[1] += entries.
__global__ void __launch_bounds__(256) count_work_kernel(CountParams p, unsigned long long *out)
{
    const uint32_t sl = blockIdx.x;
    unsigned long long segs = 0, entries = 0;
    for (uint32_t g = 0; g < p.n_groups; g++)
        for (uint32_t k = 0; k < p.n_keys; k++) {
            const KeyBins kb = p.keybins[(uint64_t)g * p.n_keys + k];
            const uint32_t n = p.placed_n[(uint64_t)sl * p.n_keys + k];
            if (g == 0) segs += (threadIdx.x == 0) ? n : 0u;
            if (kb.nbins == 0) continue;
            const uint32_t *__restrict__ soff = p.boff + kb.base;
            const uint32_t *__restrict__ coff = p.boff + p.coff_base + kb.base;
            const uint64_t *__restrict__ segl = p.placed + p.key_base[k] + (uint64_t)sl * p.sample_stride;
            for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
                const uint64_t sg = segl[i];
                const uint32_t b0 = seg_start(sg) >> kb.shift;
                if (b0 >= kb.nbins) continue;
                const uint32_t b1 = min((seg_end(sg) - 1u) >> kb.shift, kb.nbins - 1u);
                entries += (coff[b0 + 1u] - coff[b0]) + (soff[b1 + 1u] - soff[b0]);
            }
        }
    for (int d = 16; d > 0; d >>= 1) {
        segs += __shfl_xor_sync(GATB_FULL, segs, d);
        entries += __shfl_xor_sync(GATB_FULL, entries, d);
    }
    if ((threadIdx.x & 31u) == 0) {
        if (segs) atomicAdd(out, segs);
        if (entries) atomicAdd(out + 1, entries);
    }
}

void launch_count_work(cudaStream_t st, const CountParams &p, unsigned long long *out)
{
    if (p.n_samples) count_work_kernel<<<p.n_samples, 256, 0, st>>>(p, out);
}

// ---------------------------------------------------------------------------------------------------
// Grid index construction (replaces a host loop over every interval).  boff[] = S half | C half, each n_boff + 1
// slots; a key owns slots base .. base + nbins of either half.
//   1  bins_pass_kernel<false>: validate, and count the entries of every list into boff[half + base + 1 + b]
//      (S: the bin the interval starts in; C: every later bin it reaches into); bins_even_kernel rounds every
//      count up to even
//   2  ONE exclusive scan over both halves (cub): boff[half + base + 1 + b] = first slot of list b, the last
//      element = slots needed (bins_total_kernel checks it against the capacity); the C lists follow the S lists
//   3  bins_pass_kernel<true>: entry position = atomicAdd(boff[half + base + 1 + b], 1); bins_pad_kernel fills the
//      spare slot of odd lists; afterwards boff[.. + 1 + b] is the END of list b = the start of list b + 1,
//      i.e. boff[half + base + b] .. boff[half + base + b + 1] is list b
// Thread = (key, rank slot j, track): with J = the longest list on the key, slot j of a list of n intervals
// is interval j*n/J (if that differs from slot j+1's).  Consecutive threads are the same slot of consecutive
// tracks, so the threads running at any time work on one neighbourhood of the key across all tracks and
// their scattered 8-byte entry writes land in a few MB that L2 merges into full lines (thread = interval in
// list order wrote every line of the index many times: 5.4 ms instead of ~1 for 20 M intervals).
template <bool FILL>
__global__ void __launch_bounds__(256) bins_pass_kernel(BuildBinsParams p)
{
    const uint32_t k = blockIdx.y;
    const uint64_t J = p.key_jmax[k];
    const uint64_t id = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t b0 = 1, b1 = 0, x = 0, y = 0, py = 0, t = 0;       // no bins unless there is a valid interval
    uint32_t *cur_s = nullptr, *cur_c = nullptr;
    if (id < J * p.a_count) {
        const uint64_t j = id / p.a_count;
        const uint32_t a = p.a_begin + (uint32_t)(id % p.a_count);
        const uint64_t l = (uint64_t)a * p.n_keys + k;
        const uint64_t o0 = p.offs[l], n = p.offs[l + 1] - o0;
        const uint64_t r = j * n / J;
        if (r != (j + 1) * n / J) {
            const uint64_t i = o0 + r;
            const uint32_t g = a / p.ka;
            t = a % p.ka;
            const KeyBins kb = p.keybins[(uint64_t)g * p.n_keys + k];
            x = p.start[i]; y = p.end[i];
            py = r ? p.end[i - 1] : 0u;
            uint32_t err = 0;
            if (y >= 0x80000000u) err |= 1u;
            if (x >= y || py > x) err |= 2u;
            if (err) { if (!FILL) atomicOr(p.error, err); }
            else if (kb.nbins) {
                cur_s = p.boff + kb.base + 1u;
                cur_c = cur_s + p.n_boff + 1u;
                b0 = min(x >> kb.shift, kb.nbins - 1u);
                b1 = min((y - 1u) >> kb.shift, kb.nbins - 1u);
            }
        }
    }
    for (uint32_t b = b0; b <= b1; b++) {
        uint32_t *cur = (b == b0) ? cur_s : cur_c;
        if (!FILL) atomicAdd(cur + b, 1u);
        else {
            const uint64_t pos = atomicAdd(cur + b, 1u);
            if (pos < p.capacity) {
                p.cent[pos] = make_uint2(x, (min(y - x, ENTRY_LEN_MASK) << 12) | t);
                if (y - x >= ENTRY_LEN_MASK) { p.civ[pos] = make_uint2(x, y); *p.has_long = 1u; }     // only ever read for these
                p.cprev[pos] = py;
            }
        }
    }
}

// every list gets an even number of slots
__global__ void __launch_bounds__(256) bins_even_kernel(uint32_t *__restrict__ boff, uint64_t n)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) boff[i] = (boff[i] + 1u) & ~1u;
}

// after the fill: a list with an odd number of entries ends on an odd index (all lists start on even ones);
// its spare slot takes the entry that overlaps nothing
__global__ void __launch_bounds__(256) bins_pad_kernel(BuildBinsParams p)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2u * (p.n_boff + 1u)) return;
    const uint32_t v = p.boff[i];
    if (v & 1u) {
        if (v < p.capacity) { p.cent[v] = make_uint2(0x7fffffffu, 0u); p.cprev[v] = 0u; }
        p.boff[i] = v + 1u;
    }
}

// what the counting kernel reads per segment: one 16-byte record per bin b,
//   .x = start of C[b]   .y = start of S[b]   .z = |C[b]| | |S[b]| << 16   .w = |S[b..b+1]| | |S[b..b+2]| << 16
// (lengths in entries, 0xffff: does not fit -- read the offset arrays): a segment covering bins b0 .. b0 + 2 finds
// both of its runs in the record of b0
__global__ void __launch_bounds__(256) bins_rec_kernel(BuildBinsParams p)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n_boff) return;
    const uint32_t *soff = p.boff, *coff = p.boff + p.n_boff + 1u;
    const uint64_t last = p.n_boff;                 // (offsets exist up to index n_boff; lists of one key are contiguous,
    const uint32_t s0 = soff[i];                    //  lengths that run into the next key are never used: b1 < nbins)
    auto fit = [](uint32_t v) { return v < 0xffffu ? v : 0xffffu; };
    const uint32_t l0 = fit(soff[min(i + 1u, last)] - s0), l1 = fit(soff[min(i + 2u, last)] - s0), l2 = fit(soff[min(i + 3u, last)] - s0);
    p.brec[i] = make_uint4(coff[i], s0, fit(coff[i + 1u] - coff[i]) | (l0 << 16), l1 | (l2 << 16));
}

__global__ void bins_total_kernel(BuildBinsParams p)
{
    // the scan ran over both halves, 2 * (n_boff + 1) elements: the last one (a slot without a list) is the
    // number of slots all lists need
    const unsigned long long total = p.boff[2u * (p.n_boff + 1u) - 1u];
    *p.total = total;
    if (total > p.capacity) atomicOr(p.error, 4u);
    // entries `capacity`, `capacity + 1` (capacity is even) are the sentinel pair: an entry at the largest
    // coordinate overlaps no segment
    p.cent[p.capacity] = p.cent[p.capacity + 1u] = make_uint2(0x7fffffffu, 0u);
    p.cprev[p.capacity] = p.cprev[p.capacity + 1u] = 0u;
}

size_t build_bins_scan_bytes(uint64_t n_boff)
{
    size_t bytes = 0;
    cub::DeviceScan::ExclusiveSum((void *)nullptr, bytes, (uint32_t *)nullptr, (uint32_t *)nullptr, (int)(2u * (n_boff + 1u)));
    return bytes;
}

// step 1 for the tracks [p.a_begin, p.a_begin + p.a_count): may be launched per chunk of tracks as their
// intervals arrive on the device
cudaError_t launch_bins_count(cudaStream_t st, const BuildBinsParams &p)
{
    if (p.n_intervals == 0 || p.n_boff == 0 || p.jmax_all == 0 || p.a_count == 0) return cudaSuccess;
    const dim3 blocks((unsigned)(((uint64_t)p.jmax_all * p.a_count + 255) / 256), p.n_keys);
    bins_pass_kernel<false><<<blocks, 256, 0, st>>>(p);
    return cudaGetLastError();
}

// steps 2 and 3 (all tracks: p.a_begin = 0, p.a_count = n_annot)
cudaError_t launch_bins_finish(cudaStream_t st, const BuildBinsParams &p, void *scan_tmp, size_t scan_bytes)
{
    const uint64_t n2 = 2u * (p.n_boff + 1u);
    const unsigned nb = (unsigned)((n2 + 255) / 256);
    if (p.n_boff) bins_even_kernel<<<nb, 256, 0, st>>>(p.boff, n2);
    cudaError_t e = cub::DeviceScan::ExclusiveSum(scan_tmp, scan_bytes, p.boff, p.boff, (int)n2, st);
    if (e != cudaSuccess) return e;
    bins_total_kernel<<<1, 1, 0, st>>>(p);
    if (p.n_intervals && p.n_boff && p.jmax_all) {
        const dim3 blocks((unsigned)(((uint64_t)p.jmax_all * p.a_count + 255) / 256), p.n_keys);
        bins_pass_kernel<true><<<blocks, 256, 0, st>>>(p);
        bins_pad_kernel<<<nb, 256, 0, st>>>(p);
    }
    if (p.n_boff) bins_rec_kernel<<<(unsigned)((p.n_boff + 255) / 256), 256, 0, st>>>(p);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------
// K5 column statistics (gat/Engine.pyx:1635-1718, :1543-1576).  The matrix is [sample][column]: a CTA owns a
// tile of STATS_COLS adjacent columns and streams all samples; thread (c, r) = (column of the tile, row of the
// pass) reads counts[s][col0 + c] for s = r, r + STATS_ROWS, ..., so a warp reads two 64-byte runs of
// neighbouring columns per load (every 32-byte sector it touches is used in full; thread = sample with a CTA per
// column pulled a whole sector per 4-byte value).  Per-thread partials are combined over the rows in a fixed
// order, so the results are deterministic.
constexpr int STATS_COLS = 16, STATS_ROWS = 16;

struct StatsThread {
    uint32_t c, r, col;
    bool live;
};
__device__ __forceinline__ StatsThread stats_thread(const StatsParams &p)
{
    StatsThread t;
    t.c = threadIdx.x & (STATS_COLS - 1);
    t.r = threadIdx.x / STATS_COLS;
    t.col = blockIdx.x * STATS_COLS + t.c;
    t.live = t.col < p.n_cols;
    return t;
}

__device__ __forceinline__ double load_val(const StatsParams &p, uint64_t s, uint32_t col)
{
    if (p.is_float) return reinterpret_cast<const double *>(p.counts)[s * p.n_cols + col];
    return (double)reinterpret_cast<const uint32_t *>(p.counts)[s * p.n_cols + col];
}

__global__ void __launch_bounds__(STATS_COLS * STATS_ROWS) stats_pass1_kernel(StatsParams p)
{
    __shared__ unsigned long long su[5][STATS_ROWS][STATS_COLS];
    __shared__ double sd[STATS_ROWS][STATS_COLS];
    __shared__ uint32_t smm[2][STATS_ROWS][STATS_COLS];
    const StatsThread t = stats_thread(p);
    const double obs = t.live ? p.observed[t.col] : 0.0;
    const uint64_t ld = p.row_stride ? p.row_stride : p.n_cols;
    unsigned long long isum = 0, nlt = 0, neq = 0, sq_lo = 0, sq_hi = 0;
    uint32_t vmin = 0xffffffffu, vmax = 0u;
    double fsum = 0.0;
    if (t.live)
        for (uint64_t s = t.r; s < p.n_samples; s += STATS_ROWS) {
            double x;
            if (p.is_float) { x = reinterpret_cast<const double *>(p.counts)[s * ld + t.col]; fsum += x; }
            else {
                const uint32_t v = reinterpret_cast<const uint32_t *>(p.counts)[s * ld + t.col];
                const unsigned long long v2 = (unsigned long long)v * v;
                isum += v; x = (double)v;
                sq_lo += v2; sq_hi += (sq_lo < v2) ? 1ull : 0ull;       // exact sum of squares (as in stats_stream.cu)
                vmin = min(vmin, v); vmax = max(vmax, v);
            }
            nlt += (x < obs) ? 1ull : 0ull;      // searchargsorted + cmpDouble (gat/Engine.pyx:122-127, 1549-1557)
            neq += (x == obs) ? 1ull : 0ull;
        }
    su[0][t.r][t.c] = nlt; su[1][t.r][t.c] = neq; su[2][t.r][t.c] = isum; su[3][t.r][t.c] = sq_lo; su[4][t.r][t.c] = sq_hi;
    sd[t.r][t.c] = fsum;
    smm[0][t.r][t.c] = vmin; smm[1][t.r][t.c] = vmax;
    __syncthreads();
    if (t.r == 0 && t.live) {
        unsigned long long a = 0, b = 0, c = 0, lo = 0, hi = 0;
        double f = 0.0;
        for (int r = 0; r < STATS_ROWS; r++) {
            a += su[0][r][t.c]; b += su[1][r][t.c]; c += su[2][r][t.c]; f += sd[r][t.c];
            const unsigned long long l2 = su[3][r][t.c];
            lo += l2; hi += su[4][r][t.c] + ((lo < l2) ? 1ull : 0ull);
            vmin = min(vmin, smm[0][r][t.c]); vmax = max(vmax, smm[1][r][t.c]);
        }
        if (p.is_float) { p.n_lt[t.col] = a; p.n_eq[t.col] = b; p.sum[t.col] = f; return; }
        // uint32: added to the caller's sums (the CTA owns its columns, so these atomics meet no other CTA's; the low
        // word's atomic reports its own carry into the high word, whatever the order of the adds)
        atomicAdd(p.n_lt + t.col, a); atomicAdd(p.n_eq + t.col, b); atomicAdd(p.isum + t.col, c);
        const unsigned long long old = atomicAdd(p.sq_lo + t.col, lo);
        atomicAdd(p.sq_hi + t.col, hi + ((old + lo < old) ? 1ull : 0ull));
        if (p.col_min) { atomicMin(p.col_min + t.col, vmin); atomicMax(p.col_max + t.col, vmax); }
    }
}

__global__ void __launch_bounds__(STATS_COLS * STATS_ROWS) stats_pass2_kernel(StatsParams p)
{
    __shared__ double sd[STATS_ROWS][STATS_COLS];
    const StatsThread t = stats_thread(p);
    const double mean = t.live ? p.mean[t.col] : 0.0;
    double acc = 0.0;
    if (t.live)
        for (uint64_t s = t.r; s < p.n_samples; s += STATS_ROWS) {
            const double d = load_val(p, s, t.col) - mean;
            acc += d * d;
        }
    sd[t.r][t.c] = acc;
    __syncthreads();
    if (t.r == 0 && t.live) {
        double f = 0.0;
        for (int r = 0; r < STATS_ROWS; r++) f += sd[r][t.c];
        p.sumsq_dev[t.col] = f;
    }
}

// order-preserving 64-bit key of a value
__device__ __forceinline__ unsigned long long val_key(const StatsParams &p, uint64_t s, uint32_t col)
{
    if (!p.is_float) return (unsigned long long)reinterpret_cast<const uint32_t *>(p.counts)[s * p.n_cols + col];
    unsigned long long b = (unsigned long long)__double_as_longlong(reinterpret_cast<const double *>(p.counts)[s * p.n_cols + col]);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

__device__ __forceinline__ double key_val(int is_float, unsigned long long k)
{
    if (!is_float) return (double)k;
    unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)b);
}

// radix select of two order statistics per column: 8 bits per pass from the top byte
__global__ void __launch_bounds__(STATS_COLS * STATS_ROWS) stats_select_kernel(StatsParams p)
{
    __shared__ unsigned int hist[2][STATS_COLS][256];
    __shared__ unsigned long long prefix_s[2][STATS_COLS];
    __shared__ unsigned long long rank_s[2][STATS_COLS];
    const StatsThread t = stats_thread(p);
    const int top = p.is_float ? 56 : 24;
    if (threadIdx.x < 2 * STATS_COLS) {
        const int w = threadIdx.x / STATS_COLS, c = threadIdx.x % STATS_COLS;
        prefix_s[w][c] = 0; rank_s[w][c] = w ? p.rank_hi : p.rank_lo;
    }
    __syncthreads();
    for (int shift = top; shift >= 0; shift -= 8) {
        for (int i = threadIdx.x; i < 2 * STATS_COLS * 256; i += blockDim.x) (&hist[0][0][0])[i] = 0;
        __syncthreads();
        const unsigned long long pre0 = prefix_s[0][t.c], pre1 = prefix_s[1][t.c];
        const unsigned long long hmask = (shift == 56) ? 0ull : (~0ull << (shift + 8));
        if (t.live)
            for (uint64_t s = t.r; s < p.n_samples; s += STATS_ROWS) {
                const unsigned long long k = val_key(p, s, t.col);
                const unsigned int b = (unsigned int)(k >> shift) & 255u;
                if ((k & hmask) == pre0) atomicAdd(&hist[0][t.c][b], 1u);
                if ((k & hmask) == pre1) atomicAdd(&hist[1][t.c][b], 1u);
            }
        __syncthreads();
        if (threadIdx.x < 2 * STATS_COLS) {
            const int w = threadIdx.x / STATS_COLS, c = threadIdx.x % STATS_COLS;
            unsigned long long r = rank_s[w][c], cum = 0;
            int b = 0;
            for (; b < 256; b++) { if (cum + hist[w][c][b] > r) break; cum += hist[w][c][b]; }
            if (b > 255) b = 255;
            rank_s[w][c] = r - cum;
            prefix_s[w][c] |= ((unsigned long long)b << shift);
        }
        __syncthreads();
    }
    if (t.r == 0 && t.live) {
        p.q_lo[t.col] = key_val(p.is_float, prefix_s[0][t.c]);
        p.q_hi[t.col] = key_val(p.is_float, prefix_s[1][t.c]);
    }
}

__global__ void __launch_bounds__(256) compare_derive_kernel(CompareParams p)
{
    const uint64_t total = p.n_samples * p.n_pairs;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t s = i / p.n_pairs;
        const uint32_t q = (uint32_t)(i % p.n_pairs);
        // same operation order as the numpy expressions: divide, add the fold pseudo-count, divide, log, shift
        const double f1 = p.obs1[q] / (p.m1[s * p.n_cols1 + (uint32_t)p.col1[q]] + p.pseudo_count) + 0.0001;
        const double f2 = p.obs2[q] / (p.m2[s * p.n_cols2 + (uint32_t)p.col2[q]] + p.pseudo_count) + 0.0001;
        p.out[i] = log(f1 / f2) + p.delta[q];
    }
}

void launch_compare_derive(cudaStream_t st, const CompareParams &p)
{
    const uint64_t total = p.n_samples * p.n_pairs;
    if (total == 0) return;
    const unsigned blocks = (unsigned)std::min<uint64_t>((total + 255) / 256, 148u * 16u);
    compare_derive_kernel<<<blocks, 256, 0, st>>>(p);
}

// ---------------------------------------------------------------------------------------------------
// counts table text.  One CTA per column walks the samples in chunks of 256 (thread = sample); a block scan
// of the lengths (digits + separator) places every number.
__device__ __forceinline__ uint32_t decimal_digits(uint32_t v)
{
    return v < 10u ? 1u : v < 100u ? 2u : v < 1000u ? 3u : v < 10000u ? 4u : v < 100000u ? 5u : v < 1000000u ? 6u
         : v < 10000000u ? 7u : v < 100000000u ? 8u : v < 1000000000u ? 9u : 10u;
}

template <bool WRITE>
__global__ void __launch_bounds__(256) format_counts_kernel(const uint32_t *__restrict__ counts, uint64_t n_samples,
                                                            uint32_t n_cols, unsigned long long *__restrict__ col_len,
                                                            const unsigned long long *__restrict__ col_off,
                                                            char *__restrict__ text)
{
    typedef cub::BlockScan<uint32_t, 256> Scan;
    __shared__ typename Scan::TempStorage tmp;
    const uint32_t col = blockIdx.x;
    unsigned long long running = 0;                 // bytes of the samples before this chunk (block-uniform)
    char *out = WRITE ? text + col_off[col] : nullptr;
    for (uint64_t s0 = 0; s0 < n_samples; s0 += 256) {
        const uint64_t s = s0 + threadIdx.x;
        uint32_t v = 0, len = 0;
        if (s < n_samples) {
            v = counts[s * n_cols + col];
            len = decimal_digits(v) + (s + 1 < n_samples ? 1u : 0u);
        }
        uint32_t excl, total;
        Scan(tmp).ExclusiveSum(len, excl, total);
        if (WRITE && s < n_samples) {
            char *q = out + running + excl;
            uint32_t d = decimal_digits(v);
            if (s + 1 < n_samples) q[d] = ',';
            while (d) { q[--d] = (char)('0' + v % 10u); v /= 10u; }
        }
        running += total;
        __syncthreads();                            // tmp is reused by the next chunk
    }
    if (!WRITE && threadIdx.x == 0) col_len[col] = running;
}

void launch_format_counts(cudaStream_t st, const uint32_t *counts, uint64_t n_samples, uint32_t n_cols,
                          unsigned long long *col_len, const unsigned long long *col_off, char *text)
{
    if (n_cols == 0) return;
    if (text == nullptr) format_counts_kernel<false><<<n_cols, 256, 0, st>>>(counts, n_samples, n_cols, col_len, col_off, text);
    else format_counts_kernel<true><<<n_cols, 256, 0, st>>>(counts, n_samples, n_cols, col_len, col_off, text);
}

void launch_stats_pass1(cudaStream_t st, const StatsParams &p)
{
    if (p.n_cols) stats_pass1_kernel<<<(p.n_cols + STATS_COLS - 1) / STATS_COLS, STATS_COLS * STATS_ROWS, 0, st>>>(p);
}
void launch_stats_pass2(cudaStream_t st, const StatsParams &p)
{
    if (p.n_cols) stats_pass2_kernel<<<(p.n_cols + STATS_COLS - 1) / STATS_COLS, STATS_COLS * STATS_ROWS, 0, st>>>(p);
}
void launch_stats_select(cudaStream_t st, const StatsParams &p)
{
    if (p.n_cols) stats_select_kernel<<<(p.n_cols + STATS_COLS - 1) / STATS_COLS, STATS_COLS * STATS_ROWS, 0, st>>>(p);
}

}  // namespace gatb
