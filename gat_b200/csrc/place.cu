// place.cu -- K1 placement, K2 isochore->contig merge, unit preparation.  sm_100a, warp per unit.
//
// The placement loop of SamplerAnnotator.sample (gat/Engine.pyx:572-634) is sequential and
// data-dependent.  With a counter-based RNG the draws of loop turn t are a pure function of
// (seed, track, unit, sample, t), so a warp evaluates 32 consecutive turns speculatively, prefix-sums
// their overlaps, accepts the turns before the first one whose length satisfies `remaining <= length`
// (gat/Engine.pyx:582) and then runs that turn's checkpoint (sort + merge(0) + workspace coverage)
// cooperatively.  (Keeping the 32 drawn turns as a window that is consumed across checkpoints was measured and
// dropped: late turns are `certain` ones whose draw is already put off, so it saved nothing and cost registers.)  The result is bit-identical to the sequential restatement in oracle/gat_oracle.c
// driven by the same Philox stream (tests/test_gpu_parity.py).
#include "place.cuh"

namespace gatb {

// ---------------------------------------------------------------------------------------------------
// draws of one loop turn (RNG contract, DESIGN.md)
struct TurnDraw { uint32_t L, start, end; int32_t ov; };

__device__ __forceinline__ uint32_t ws_pick(const WsView &w, uint32_t r)
{
    // first i with cuminc[i] > r   == searchsorted(cdf, r) with cdf = cuminc - 1 (gat/Engine.pyx:300-305)
    if (w.n == 1) return 0;
    uint32_t lo = 0, hi = w.n;
    if (w.tabw != nullptr) {                // bucket table: the answer lies in [tab[b], tab[b + 1]]
        const uint32_t b = __umulhi(r, w.tabw[0]);
        const uint16_t *t = ws_tab16(w);
        lo = t[b]; hi = t[b + 1u];
    }
    while (lo < hi) {
        uint32_t mid = (lo + hi) >> 1;
        if (w.cuminc[mid] > r) hi = mid; else lo = mid + 1;
    }
    return lo;
}

__device__ __forceinline__ TurnDraw draw_turn(const UnitDesc &d, const WsView &ws, const uint32_t *tab,
                                              uint32_t turn, uint32_t c1base, uint32_t unit, uint32_t sample,
                                              const PhiloxKeys &rk)
{
    Philox4 b0 = philox4x32_10(turn, 0u | c1base, unit, sample, rk);
    Philox4 b1 = philox4x32_10(turn, 1u | c1base, unit, sample, rk);
    TurnDraw t;
    // HistogramSampler.sample (gat/Engine.pyx:413-435): r = randint(1,total) ranks the sorted lengths
    uint32_t r = 1;
    if (d.tab_n > 1) r = 1 + bounded_u32(b0.x, b0.y, d.tab_n - 1);
    uint32_t L = tab[r - 1];
    if (d.bucket > 1) L += bounded_u32(b1.z, b1.w, d.bucket);
    t.L = L;
    // SegmentListSampler.sample (gat/Engine.pyx:279-348)
    uint32_t rw = bounded_u32(b0.z, b0.w, d.ws_total);
    uint32_t i = ws_pick(ws, rw);
    uint32_t cs = ws.start[i], ce = ws.end[i];
    int64_t sstart = (int64_t)cs - (int64_t)L + 1;
    if (i > 0) sstart = (int64_t)max((int32_t)ws.end[i - 1], (int32_t)sstart);
    uint32_t range = (uint32_t)((int64_t)ce - sstart);
    int64_t pp = sstart + (int64_t)bounded_u32(b1.x, b1.y, range);
    t.start = (uint32_t)max(0, (int32_t)pp);
    t.end = (uint32_t)(pp + (int64_t)L);
    t.ov = max(0, min((int32_t)ce, (int32_t)t.end) - max((int32_t)cs, (int32_t)t.start));
    return t;
}

// SegmentList._getInsertionPoint (gat/SegmentList.pyx:853-887) on packed segments
__device__ __forceinline__ int insertion_point(const uint64_t *buf, uint32_t n, uint32_t ostart, uint32_t oend)
{
    if (n == 0) return -1;
    if (ostart >= seg_end(buf[n - 1])) return (int)n;
    if (oend <= seg_start(buf[0])) return -1;
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        uint32_t mid = lo + ((hi - lo) >> 1);
        if (((int32_t)seg_start(buf[mid]) - (int32_t)ostart) < 0) lo = mid + 1; else hi = mid;
    }
    if (lo == n) return (int)lo - 1;
    if (seg_start(buf[lo]) != ostart) return (int)lo - 1;
    return (int)lo;
}

// overshoot repair (gat/Engine.pyx:608-625): SegmentListSampler(U).sample(1) picks a base of U,
// trim_ends (gat/SegmentList.pyx:545-597) removes `size` bases from that segment's start or end
// -> *removed = workspace bases the trim took away, *emptied = segments it left empty, *orphaned = segments
// it left non-empty but without a base in the workspace
// `total` = total length of U (kept by the caller from checkpoint to checkpoint)
__device__ __forceinline__ void warp_trim(uint64_t *buf, uint32_t nu, uint32_t size, uint32_t total,
                                          const Philox4 &b2, const Philox4 &b3, const WsView &ws,
                                          uint32_t *removed, uint32_t *emptied, uint32_t *orphaned)
{
    const int lane = lane_id();
    uint32_t rem = 0, emp = 0, orph = 0;
    uint32_t r = bounded_u32(b2.x, b2.y, total);
    // first idx with inclusive cumulative length > r
    uint32_t running = 0, idx = nu;
    for (uint32_t b0 = 0; b0 < nu; b0 += 32) {
        uint32_t i = b0 + lane;
        uint32_t len = 0;
        if (i < nu) { uint64_t x = buf[i]; len = seg_end(x) - seg_start(x); }
        uint32_t incl = warp_incl_scan_add_u32(len);
        uint32_t m = __ballot_sync(GATB_FULL, (i < nu) && (running + incl > r));
        if (m) { idx = b0 + (uint32_t)__ffs(m) - 1; break; }
        running += __shfl_sync(GATB_FULL, incl, 31);
    }
    if (lane == 0 && idx < nu) {
        uint64_t x = buf[idx];
        uint32_t cs = seg_start(x), ce = seg_end(x);
        int64_t sstart = (int64_t)cs - 1 + 1;
        if (idx > 0) sstart = (int64_t)max((int32_t)seg_end(buf[idx - 1]), (int32_t)sstart);
        uint32_t range = (uint32_t)((int64_t)ce - sstart);
        int64_t pp = sstart + (int64_t)bounded_u32(b2.z, b2.w, range);
        uint32_t pos = (uint32_t)max(0, (int32_t)pp);
        int forward = (int)bounded_u32(b3.x, b3.y, 2u);
        int32_t sz = (int32_t)size;
        int k = insertion_point(buf, nu, pos, pos + 1);
        if (k == (int)nu) k = 0;
        if (k < 0) k = (int)nu - 1;
        while (sz > 0) {
            uint64_t y = buf[k];
            int32_t l = (int32_t)seg_end(y) - (int32_t)seg_start(y);
            const uint32_t before = ws_overlap(ws, seg_start(y), seg_end(y));
            if (l < sz) { buf[k] = 0; sz -= l; rem += before; emp += (l > 0) ? 1u : 0u; }
            else {
                uint64_t z;
                if (forward) z = pack_seg(seg_start(y) + (uint32_t)sz, seg_end(y));
                else z = pack_seg(seg_start(y), (uint32_t)((int32_t)seg_end(y) - sz));
                buf[k] = z;
                const uint32_t after = ws_overlap(ws, seg_start(z), seg_end(z));
                rem += before - after;
                emp += (l == sz) ? 1u : 0u;
                orph += (l != sz && after == 0u) ? 1u : 0u;
                sz = 0;
            }
            if (forward) { k += 1; if (k == (int)nu) k = 0; }
            else { k -= 1; if (k < 0) k = (int)nu - 1; }
        }
    }
    __syncwarp();
    *removed = __shfl_sync(GATB_FULL, rem, 0);
    *emptied = __shfl_sync(GATB_FULL, emp, 0);
    *orphaned = __shfl_sync(GATB_FULL, orph, 0);
}

// ONE new segment behind a sorted, merged list (the usual late checkpoint): when it touches neither
// neighbour, merge(0) of the whole amounts to sliding it into place.  false: it does touch one (the general
// insert-and-merge path takes over, nothing was changed).
__device__ __forceinline__ bool warp_insert_one(uint64_t *buf, uint32_t &nu, const WsView &ws, uint32_t &cov,
                                                uint32_t &ulen)
{
    const int lane = lane_id();
    const uint64_t key = buf[nu];
    const uint32_t xs = seg_start(key), xe = seg_end(key);
    if (xs == xe) return true;                      // empty: merge(0) drops it
    uint32_t lo = 0, hi = nu;                       // elements with key <= the new one (same probes in every lane)
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (buf[mid] <= key) lo = mid + 1; else hi = mid;
    }
    const uint32_t pos = lo;
    if (pos > 0 && seg_end(buf[pos - 1]) >= xs) return false;       // overlaps or touches its left neighbour
    if (pos < nu && xe >= seg_start(buf[pos])) return false;        // ... its right neighbour
    __syncwarp();
    if (nu > pos) {
        for (int c = (int)((nu - 1) >> 5); c >= (int)(pos >> 5); c--) {     // slide up by one, top chunk first
            const uint32_t i = ((uint32_t)c << 5) + lane;
            const uint64_t x = (i < nu) ? buf[i] : 0;
            __syncwarp();
            if (i < nu && i >= pos) buf[i + 1] = x;
            __syncwarp();
        }
    }
    if (lane == 0) buf[pos] = key;
    __syncwarp();
    nu += 1;
    cov += ws_overlap(ws, xs, xe);
    ulen += xe - xs;
    return true;
}

// keep segments overlapping the workspace by >= 1 base (SegmentList.filter, gat/SegmentList.pyx:1401-1467)
__device__ __forceinline__ uint32_t warp_filter_ws(uint64_t *buf, uint32_t n, const WsView &ws)
{
    const int lane = lane_id();
    uint32_t nout = 0;
    for (uint32_t b0 = 0; b0 < n; b0 += 32) {
        uint32_t i = b0 + lane;
        uint64_t x = (i < n) ? buf[i] : 0;
        bool keep = (i < n) && (ws_overlap(ws, seg_start(x), seg_end(x)) > 0);
        uint32_t m = __ballot_sync(GATB_FULL, keep);
        __syncwarp();
        if (keep) buf[nout + __popc(m & ((1u << lane) - 1))] = x;
        nout += __popc(m);
        __syncwarp();
    }
    return nout;
}

// After trim_ends the list is still sorted and merged (segments only shrank or were emptied, and
// merge(0) had left a gap between neighbours), so sort + merge(0) reduces to dropping the empty segments.
// *cov = workspace coverage of what is left (the segments are disjoint).
__device__ __forceinline__ uint32_t warp_drop_empty(uint64_t *buf, uint32_t n, const WsView &ws, uint32_t *cov)
{
    const int lane = lane_id();
    uint32_t nout = 0, covered = 0;
    for (uint32_t b0 = 0; b0 < n; b0 += 32) {
        uint32_t i = b0 + lane;
        uint64_t x = (i < n) ? buf[i] : 0;
        bool keep = (i < n) && (seg_start(x) != seg_end(x));
        if (keep) covered += ws_overlap(ws, seg_start(x), seg_end(x));
        uint32_t m = __ballot_sync(GATB_FULL, keep);
        __syncwarp();
        if (keep) buf[nout + __popc(m & ((1u << lane) - 1))] = x;
        nout += __popc(m);
        __syncwarp();
    }
    *cov = __reduce_add_sync(GATB_FULL, covered);
    return nout;
}

// ---------------------------------------------------------------------------------------------------
// K1: one warp per (unit, sample)
#ifndef GATB_PLACE_MINBLOCKS
#define GATB_PLACE_MINBLOCKS 8      // 64 registers: occupancy beats the few spilled values (measured)
#endif
// ONE_PIECE: every unit's workspace is one piece (contig workspaces, PlaceParams.one_piece).  With the piece count a
// constant the compiler drops the piece draw, its search, the predecessor clamp and the multi-piece branches of the
// coverage helpers from every turn.
template <bool ONE_PIECE>
__global__ void __launch_bounds__(128, GATB_PLACE_MINBLOCKS) place_kernel(PlaceParams p)
{
    __shared__ uint32_t sort_cnt[4][GATB_SORT_NB];         // counting-sort buckets, one set per warp
    const uint64_t item = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (item >= (uint64_t)p.n_units * p.n_samples) return;
    const int lane = lane_id();
    uint32_t *cnt = sort_cnt[threadIdx.x >> 5];
    const uint32_t unit = p.order[item / p.n_samples];
    const uint32_t sl = (uint32_t)(item % p.n_samples);
    const UnitDesc d = p.units[unit];
    uint64_t *buf = p.buf + (uint64_t)sl * p.sample_stride + d.buf_off;
    WsView ws;
    ws.start = p.ws_start + d.ws_off; ws.end = p.ws_end + d.ws_off; ws.cuminc = p.ws_cuminc + d.ws_off;
    ws.n = ONE_PIECE ? 1u : d.ws_n;
    ws.tabw = !ONE_PIECE && d.ws_tab_off != 0xffffffffu ? p.ws_tab + d.ws_tab_off : nullptr;
    const uint32_t *tab = p.len_tab + d.tab_off;
    const uint32_t sample = (uint32_t)(p.sample_begin + sl);
    const uint32_t c1base = p.track << 8;

    // every placement starts in [first workspace start - longest length, last workspace end): the range of
    // the counting sort's buckets, known without a pass over the keys
    // (and as many placements as segments are expected): the sort's plan is fixed now, and the bulk phase
    // counts every placement it accepts into the plan's buckets, so the first checkpoint's sort starts with
    // its histogram done
    SortPlan plan;
    plan.lo = 0; plan.inv = 0; plan.nb = 0;
    bool prehist = false;
    if (d.tab_n > 0) {
        plan.lo = d.plan_lo; plan.inv = d.plan_inv; plan.nb = d.plan_nb;       // (sample-invariant: prep_units_kernel)
        for (uint32_t b = lane; b < plan.nb; b += 32) cnt[b] = 0u;
        __syncwarp();
        prehist = p.sampler_kind == 0;
    }
    int32_t remaining = d.ltotal, true_remaining = d.ltotal;
    int fails = 0;
    uint32_t nu = 0, np = 0, t0 = 0, status = 0;
    uint32_t cov = 0;                   // workspace coverage of buf[0,nu) as of the last checkpoint / trim
    uint32_t ulen = 0;                  // its total length
    uint32_t trim_emptied = 0;          // segments the last trim left empty
    uint32_t orphans = 0;               // segments any trim left outside the workspace
    bool dirty = false;

    if (d.tab_n > 0 && p.sampler_kind == 1 && d.seg_n > d.cap) status |= UNIT_OVERFLOW;
    else if (d.tab_n > 0 && p.sampler_kind == 1) {
        // SamplerSegments.sample (gat/Engine.pyx:719-735): exactly len(segments) placements, every one
        // kept, returned in draw order (unsorted, unmerged); fromIsochores' merge(0) normalizes them later
        for (uint32_t t = lane; t < d.seg_n; t += 32) {
            const TurnDraw td = draw_turn(d, ws, tab, t, c1base, unit, sample, p.keys);
            buf[t] = pack_seg(td.start, td.end);
        }
        nu = d.seg_n;
        __syncwarp();
    } else if (d.tab_n > 0) {
        while (true_remaining > 0 && fails < 20) {
            // ---- speculative batch of 32 turns ------------------------------------------------------
            // (remaining <= 0: turn t0 triggers the checkpoint whatever its length, so its draw is put
            // off until the checkpoint has shown that the turn is placed at all -- usually it is not)
            const bool certain = remaining <= 0;
            TurnDraw t;
            t.L = 0; t.start = 0; t.end = 0; t.ov = 0;
            uint32_t f = 0;
            int32_t incl = 0;
            if (!certain) {
                t = draw_turn(d, ws, tab, t0 + lane, c1base, unit, sample, p.keys);
                // no turn can trigger while what is left after ALL 32 still exceeds the longest of their lengths
                // (two warp reductions instead of the prefix scan: the usual case until the unit is nearly full)
                const int32_t all = __reduce_add_sync(GATB_FULL, t.ov);
                if (remaining - all > (int32_t)__reduce_max_sync(GATB_FULL, t.L)) {
                    f = 32u;
                    incl = all;                     // (only lane 31's value is read below)
                } else {
                    incl = warp_incl_scan_add(t.ov);
                    int32_t rem_before = remaining - (incl - t.ov);
                    uint32_t trig = __ballot_sync(GATB_FULL, rem_before <= (int32_t)t.L);
                    f = trig ? (uint32_t)__ffs(trig) - 1 : 32u;
                }
            }
            if (nu + np + f + 1 > d.cap) {
                // buffer full: merge now.  merge(0) is idempotent and associative on the set of
                // accepted placements, so an early merge does not change any later result.
                __syncwarp();
                nu = warp_sort_merge0(buf, nu + np, nullptr, nullptr, &ws, &cov, &ulen);
                np = 0; dirty = false; prehist = false;
                if (nu + 33 > d.cap) { status |= UNIT_OVERFLOW; break; }
            }
            if ((uint32_t)lane < f) {
                buf[nu + np + lane] = pack_seg(t.start, t.end);
                if (prehist) atomicAdd(&cnt[sort_bucket(plan, t.start)], 1u);
            }
            if (f > 0) remaining -= __shfl_sync(GATB_FULL, incl, (int)f - 1);
            np += f; t0 += f;
            if (f == 32) continue;

            // ---- turn t0: `remaining <= length` -> checkpoint (gat/Engine.pyx:582-605) ---------------
            uint32_t sf = __shfl_sync(GATB_FULL, t.start, (int)f);
            uint32_t ef = __shfl_sync(GATB_FULL, t.end, (int)f);
            int32_t ovf = __shfl_sync(GATB_FULL, t.ov, (int)f);
            __syncwarp();
            // late checkpoints add a handful of placements to an already merged list: insert them
            // instead of re-sorting everything (same result, see warp_insert_merge0)
            // the merge pass of every variant also returns the workspace coverage of the merged list
            if (dirty && np == 0) {                 // straight after a trim: still sorted and merged
                if (trim_emptied) nu = warp_drop_empty(buf, nu, ws, &cov);
            } else if (nu > 0 && np == 1 && !dirty && warp_insert_one(buf, nu, ws, cov, ulen)) {
            } else if (nu > 0 && np < 32 && !dirty) nu = warp_insert_merge0(buf, nu, np, &ws, &cov, &ulen);
            else {
                const uint32_t n = nu + np;         // the free upper part of the buffer is the sort's scratch
                nu = warp_sort_merge0(buf, n, 2u * n <= d.cap ? buf + n : nullptr, cnt, &ws, &cov, &ulen,
                                      &plan, prehist && nu == 0);
                prehist = false;
            }
            np = 0; dirty = false;
            remaining = d.ltotal - (int32_t)cov;
            if (true_remaining == remaining) fails++; else true_remaining = remaining;

            if (true_remaining < 0) {           // overshoot (gat/Engine.pyx:608-625)
                Philox4 b2 = philox4x32_10(t0, 2u | c1base, unit, sample, p.keys);
                Philox4 b3 = philox4x32_10(t0, 3u | c1base, unit, sample, p.keys);
                uint32_t removed, orphaned;
                warp_trim(buf, nu, (uint32_t)(-true_remaining), ulen, b2, b3, ws, &removed, &trim_emptied, &orphaned);
                cov -= removed; orphans += orphaned;
                ulen -= (uint32_t)(-true_remaining);
                dirty = true;
                true_remaining = 1;
                t0 += 1;
                continue;
            }
            if (true_remaining > 0) {           // gat/Engine.pyx:632-634
                if (certain) {                  // the draw that was put off (every lane computes turn t0)
                    const TurnDraw t1 = draw_turn(d, ws, tab, t0, c1base, unit, sample, p.keys);
                    sf = t1.start; ef = t1.end; ovf = t1.ov;
                }
                if (lane == 0) buf[nu + np] = pack_seg(sf, ef);
                np += 1;
                remaining -= ovf;
            }
            t0 += 1;
        }
        if (fails >= 20) status |= UNIT_HIT_ROUND_CAP;
        // result = unintersected.merge(0).filter(workspace) (gat/Engine.pyx:639-646); placements
        // still pending (appended after the last checkpoint) are dropped, as in the reference
        __syncwarp();
        if (dirty && trim_emptied) nu = warp_drop_empty(buf, nu, ws, &cov);
        // every placement has a base in the workspace piece it was drawn for, hence so has every merged
        // segment: only a trim can have left one outside
        if (orphans) nu = warp_filter_ws(buf, nu, ws);
    }
    __syncwarp();
    if (lane == 0) {
        uint32_t slot = p.out_by_contig ? d.contig : unit;
        p.out_n[(uint64_t)sl * p.out_n_stride + slot] = (status & UNIT_OVERFLOW) ? 0u : nu;
        if (p.status) p.status[(uint64_t)sl * p.n_units + unit] = (uint8_t)status;
        if ((status & UNIT_OVERFLOW) && p.unit_over) p.unit_over[unit] = 1u;
    }
}

// ---------------------------------------------------------------------------------------------------
// SamplerShift.sample (gat/Engine.pyx:998-1111): every workspace-overlapping segment is moved to a random
// position of the workspace within +-shift_area of its midpoint and wrapped around the ends of that local
// workspace.  Segments are independent of each other: one warp per (unit, sample), lane = segment; the
// pieces go to the unit buffer through a per-warp counter, then the warp sorts and normalizes them (:1109).
// The uint32 / int32 conversions of the Cython code are kept (oracle/gat_oracle.c:go_sampler_shift).

// workspace pieces clipped to the window [w0, w1): getOverlappingSegmentsWithRange + truncate
// (gat/SegmentList.pyx:957-985, 1186-1202); the clipped pieces are never empty
struct LocalWs {
    const uint32_t *ws_s, *ws_e;
    uint32_t k, w0, w1;
    __device__ __forceinline__ uint32_t s(uint32_t i) const { return max(ws_s[i], w0); }
    __device__ __forceinline__ uint32_t e(uint32_t i) const { return min(ws_e[i], w1); }
};

// _getInsertionPoint(Segment(x, x + 1)) on the local workspace (gat/SegmentList.pyx:853-887) with the
// border fix of its callers (:1336-1337)
__device__ __forceinline__ uint32_t local_insertion_point(const LocalWs &L, uint32_t x)
{
    if (x >= L.e(L.k - 1u)) return L.k - 1u;
    if (x + 1u <= L.s(0)) return 0u;
    uint32_t lo = 0, hi = L.k;
    while (lo < hi) {                       // first piece with start >= x
        const uint32_t mid = (lo + hi) >> 1;
        if (L.s(mid) < x) lo = mid + 1; else hi = mid;
    }
    if (lo == L.k || L.s(lo) != x) return lo - 1u;      // (lo >= 1 here: x + 1 > s(0) and s(0) != x)
    return lo;
}

struct PieceSink {
    uint64_t *buf;
    uint32_t *counter;
    uint32_t cap;
    __device__ __forceinline__ void operator()(uint32_t s, uint32_t e) const
    {
        if (s == e) return;                 // (normalize drops empty segments)
        const uint32_t pos = atomicAdd(counter, 1u);
        if (pos < cap) buf[pos] = pack_seg(s, e);
    }
};

// getFilledSegmentsFromStart (gat/SegmentList.pyx:1314-1355)
__device__ __forceinline__ void fill_from_start(const LocalWs &L, uint32_t total, uint32_t start, int32_t remainder,
                                                const PieceSink &emit)
{
    if ((uint32_t)remainder > total) {
        for (uint32_t i = 0; i < L.k; i++) emit(L.s(i), L.e(i));
        return;
    }
    uint32_t idx = local_insertion_point(L, start);
    for (uint32_t it = 0; remainder > 0 && it < 2u * L.k + 4u; it++) {      // (the walk ends within two rounds)
        const uint32_t ps = L.s(idx), pe = L.e(idx);
        if (!(pe < start)) {
            start = (uint32_t)max((int32_t)ps, (int32_t)start);
            const uint32_t end = (uint32_t)min((int32_t)pe, (int32_t)(start + (uint32_t)remainder));
            remainder -= (int32_t)(end - start);
            emit(start, end);
        }
        idx += 1;
        if (idx == L.k) { idx = 0; start = L.s(0); }
    }
}

// getFilledSegmentsFromEnd (gat/SegmentList.pyx:1357-1399)
__device__ __forceinline__ void fill_from_end(const LocalWs &L, uint32_t total, uint32_t end, int32_t remainder,
                                              const PieceSink &emit)
{
    if ((uint32_t)remainder > total) {
        for (uint32_t i = 0; i < L.k; i++) emit(L.s(i), L.e(i));
        return;
    }
    uint32_t idx = local_insertion_point(L, end);
    for (uint32_t it = 0; remainder > 0 && it < 2u * L.k + 4u; it++) {
        const uint32_t ps = L.s(idx), pe = L.e(idx);
        if (!(ps > end)) {
            end = (uint32_t)min((int32_t)pe, (int32_t)end);
            const uint32_t start = (uint32_t)max((int32_t)ps, (int32_t)(end - (uint32_t)remainder));
            remainder -= (int32_t)(end - start);
            emit(start, end);
        }
        if (idx == 0) { idx = L.k - 1u; end = L.e(idx); } else idx -= 1;
    }
}

__global__ void __launch_bounds__(128) shift_kernel(PlaceParams p)
{
    __shared__ uint32_t sort_cnt[4][GATB_SORT_NB];
    __shared__ uint32_t emitted[4];
    const uint64_t item = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (item >= (uint64_t)p.n_units * p.n_samples) return;
    const int lane = lane_id();
    const uint32_t unit = p.order[item / p.n_samples];
    const uint32_t sl = (uint32_t)(item % p.n_samples);
    const UnitDesc d = p.units[unit];
    uint64_t *buf = p.buf + (uint64_t)sl * p.sample_stride + d.buf_off;
    WsView ws;
    ws.start = p.ws_start + d.ws_off; ws.end = p.ws_end + d.ws_off; ws.cuminc = p.ws_cuminc + d.ws_off;
    ws.n = d.ws_n;
    ws.tabw = d.ws_tab_off != 0xffffffffu ? p.ws_tab + d.ws_tab_off : nullptr;
    const uint32_t sample = (uint32_t)(p.sample_begin + sl);
    const uint32_t c1 = p.track << 8;       // Philox block 0 of turn x: words 0,1 = position, words 2,3 = direction
    uint32_t *counter = &emitted[threadIdx.x >> 5];
    if (lane == 0) *counter = 0u;
    __syncwarp();
    PieceSink emit;
    emit.buf = buf; emit.counter = counter; emit.cap = d.cap;
    const uint32_t *ss = p.seg_start + d.seg_off, *se = p.seg_end + d.seg_off;

    uint32_t nw = 0;                        // working segments so far = segments.filter(workspace) (:1060-1062)
    for (uint32_t b0 = 0; b0 < d.seg_n; b0 += 32) {
        const uint32_t i = b0 + lane;
        uint32_t s = 0, e = 0;
        bool keep = false;
        if (i < d.seg_n) { s = ss[i]; e = se[i]; keep = ws_overlap(ws, s, e) > 0; }
        const uint32_t m = __ballot_sync(GATB_FULL, keep);
        const uint32_t x = nw + __popc(m & ((1u << lane) - 1));      // index in the working list = Philox turn
        nw += __popc(m);
        if (!keep) continue;
        const uint32_t length = e - s, midpoint = s + length / 2u;
        int32_t shift_area;
        if (p.shift_extension) shift_area = p.shift_extension / 2;                       // :1074-1077
        else shift_area = (int32_t)(uint32_t)floor((double)length * p.shift_half_radius);
        const int32_t w0 = max(0, (int32_t)(midpoint - (uint32_t)shift_area));          // :1080-1081
        const int32_t w1 = max(0, (int32_t)(midpoint + (uint32_t)shift_area));
        if (w0 >= w1) continue;             // empty window: the segment drops out (see below)
        // pieces of the window: from the first one ending after w0 to the last one starting before w1
        uint32_t lo = 0, hi = ws.n;
        while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (ws.end[mid] > (uint32_t)w0) hi = mid; else lo = mid + 1; }
        const uint32_t first = lo;
        hi = ws.n;
        while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (ws.start[mid] >= (uint32_t)w1) hi = mid; else lo = mid + 1; }
        LocalWs L;
        L.ws_s = ws.start + first; L.ws_e = ws.end + first; L.k = lo - first; L.w0 = (uint32_t)w0; L.w1 = (uint32_t)w1;
        // No workspace in the window: numpy.random.randint(0, 0) raises inside the cpdef getRandomPosition,
        // whose C return type cannot carry the exception -- it is ignored, 0 comes back and every fill of the
        // empty local workspace returns nothing: the segment silently drops out of the sample
        if (L.k == 0) continue;
        uint32_t total = 0;
        for (uint32_t j = 0; j < L.k; j++) total += L.e(j) - L.s(j);
        const Philox4 r = philox4x32_10(x, c1, unit, sample, p.keys);
        uint32_t pos = bounded_u32(r.x, r.y, total);                  // getRandomPosition (gat/SegmentList.pyx:902-915)
        int32_t start = 0, end;
        for (uint32_t j = 0; j < L.k; j++) {
            const uint32_t l = L.e(j) - L.s(j);
            if (pos > l) pos -= l;
            else { start = (int32_t)(L.s(j) + pos); break; }
        }
        if (bounded_u32(r.z, r.w, 2u)) end = (int32_t)((uint32_t)start + length);       // :1086-1090
        else { end = start; start = (int32_t)((uint32_t)end - length); }
        const int32_t lws = (int32_t)L.s(0), lwe = (int32_t)L.e(L.k - 1u);              // :1093 ws.min(), ws.max()
        // one forward and one backward fill at most; their order does not matter (the pieces are sorted later)
        // and a fill of 0 bases returns nothing, so each walk is instantiated once in the kernel
        uint32_t fs_start, fe_end = 0;
        int32_t fs_rem, fe_rem = 0;
        if (start < lws) {                                                               // :1096-1100
            const int32_t remainder = min(lws - start, (int32_t)length);
            fs_start = (uint32_t)start; fs_rem = (int32_t)(length - (uint32_t)remainder);
            fe_end = (uint32_t)lwe; fe_rem = remainder;
        } else if (end > lwe) {                                                          // :1101-1105
            const int32_t remainder = min(end - lwe, (int32_t)length);
            fe_end = (uint32_t)end; fe_rem = (int32_t)(length - (uint32_t)remainder);
            fs_start = (uint32_t)lws; fs_rem = remainder;
        } else { fs_start = (uint32_t)start; fs_rem = (int32_t)length; }                // :1107
        if (fs_rem > 0) fill_from_start(L, total, fs_start, fs_rem, emit);
        if (fe_rem > 0) fill_from_end(L, total, fe_end, fe_rem, emit);
    }
    __syncwarp();
    const uint32_t n = *counter;
    uint32_t status = 0, nu = 0;
    if (n > d.cap) status |= UNIT_OVERFLOW;
    else nu = warp_sort_merge0<true>(buf, n, 2u * n <= d.cap ? buf + n : nullptr, sort_cnt[threadIdx.x >> 5]);
    __syncwarp();
    if (lane == 0) {
        const uint32_t slot = p.out_by_contig ? d.contig : unit;
        p.out_n[(uint64_t)sl * p.out_n_stride + slot] = nu;
        if (p.status) p.status[(uint64_t)sl * p.n_units + unit] = (uint8_t)status;
        if ((status & UNIT_OVERFLOW) && p.unit_over) p.unit_over[unit] = 1u;
    }
}

void launch_place(cudaStream_t st, const PlaceParams &p)
{
    uint64_t items = (uint64_t)p.n_units * p.n_samples;
    if (items == 0) return;
    const int warps_per_block = 4;
    uint64_t blocks = (items + warps_per_block - 1) / warps_per_block;
    if (p.sampler_kind == 2) shift_kernel<<<(unsigned)blocks, warps_per_block * 32, 0, st>>>(p);
    else if (p.one_piece) place_kernel<true><<<(unsigned)blocks, warps_per_block * 32, 0, st>>>(p);
    else place_kernel<false><<<(unsigned)blocks, warps_per_block * 32, 0, st>>>(p);
}

// ---------------------------------------------------------------------------------------------------
// K2: IntervalDictionary.fromIsochores (gat/Engine.pyx:2857-2876): per contig, extend with every
// isochore unit's list (unit order) then merge(0).  One warp per (contig, sample).
__global__ void __launch_bounds__(128) contig_merge_kernel(MergeParams p)
{
    __shared__ uint32_t sort_cnt[4][GATB_SORT_NB];
    const uint64_t item = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (item >= (uint64_t)p.n_contigs * p.n_samples) return;
    const int lane = lane_id();
    const uint32_t c = (uint32_t)(item / p.n_samples);
    const uint32_t sl = (uint32_t)(item % p.n_samples);
    uint64_t *dst = p.placed + (uint64_t)sl * p.placed_stride + p.contig_base[c];
    uint32_t total = 0;
    for (uint32_t k = p.contig_unit_off[c]; k < p.contig_unit_off[c + 1]; k++) {
        uint32_t u = p.contig_units[k];
        uint32_t n = p.unit_n[(uint64_t)sl * p.n_units + u];
        const uint64_t *src = p.unit_buf + (uint64_t)sl * p.unit_stride + p.units[u].buf_off;
        for (uint32_t i = lane; i < n; i += 32) dst[total + i] = src[i];
        total += n;
    }
    __syncwarp();
    const uint64_t cap = (c + 1 < p.n_contigs ? p.contig_base[c + 1] : p.placed_stride) - p.contig_base[c];
    uint32_t n = warp_sort_merge0(dst, total, 2ull * total <= cap ? dst + total : nullptr, sort_cnt[threadIdx.x >> 5]);
    __syncwarp();
    if (lane == 0) p.placed_n[(uint64_t)sl * p.n_contigs + c] = n;
}

void launch_contig_merge(cudaStream_t st, const MergeParams &p)
{
    uint64_t items = (uint64_t)p.n_contigs * p.n_samples;
    if (items == 0) return;
    const int warps_per_block = 4;
    uint64_t blocks = (items + warps_per_block - 1) / warps_per_block;
    contig_merge_kernel<<<(unsigned)blocks, warps_per_block * 32, 0, st>>>(p);
}

// ---------------------------------------------------------------------------------------------------
// Sample-invariant preparation of every unit (gat/Engine.pyx:543-565), one warp per unit:
//   working = segments.filter(workspace); ltotal = working.intersect(workspace).sum();
//   histogram of ceil(len/bucket) (gat/SegmentList.pyx:1148-1184) kept as the sorted table
//   tab[r-1] = bucket_index * bucket, which is what lower_bound(cdf, r) * bucket returns
//   (gat/Engine.pyx:424-430) without materialising the 100000-bucket CDF.
__global__ void __launch_bounds__(128) prep_units_kernel(UnitDesc *units, uint32_t n_units,
                                                         const uint32_t *seg_start, const uint32_t *seg_end,
                                                         const uint32_t *ws_start, const uint32_t *ws_end,
                                                         const uint32_t *ws_cuminc, uint32_t *len_tab,
                                                         uint64_t *scratch, const uint64_t *scratch_off,
                                                         uint32_t bucket_size, uint32_t nbuckets, uint32_t *ws_tab)
{
    const uint32_t unit = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (unit >= n_units) return;
    const int lane = lane_id();
    UnitDesc d = units[unit];
    WsView ws;
    ws.start = ws_start + d.ws_off; ws.end = ws_end + d.ws_off; ws.cuminc = ws_cuminc + d.ws_off; ws.n = d.ws_n;
    ws.tabw = nullptr;
    // bucket tables over the unit's workspace pieces (common.cuh), for units with enough pieces to search
    if (d.ws_tab_off != 0xffffffffu) {
        const uint32_t first = ws.start[0], span = ws.end[ws.n - 1u] - first;
        const uint32_t pick_inv = (uint32_t)min(((unsigned long long)WS_NB << 32) / d.ws_total, 0xffffffffull);
        const uint32_t end_inv = (uint32_t)min(((unsigned long long)WS_NB << 32) / span, 0xffffffffull);
        uint32_t *tw = ws_tab + d.ws_tab_off;
        uint16_t *t = reinterpret_cast<uint16_t *>(tw + 2);
        if (lane == 0) { tw[0] = pick_inv; tw[1] = end_inv; }
        for (uint32_t b = lane; b <= WS_NB; b += 32) {
            // smallest value of bucket b (or something below it): floor(b * 2^32 / inv)
            const unsigned long long r = min(((unsigned long long)b << 32) / pick_inv, (unsigned long long)d.ws_total - 1ull);
            uint32_t lo = 0, hi = ws.n;
            while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (ws.cuminc[mid] > (uint32_t)r) hi = mid; else lo = mid + 1; }
            t[b] = (uint16_t)(b == WS_NB ? ws.n - 1u : lo);
            const unsigned long long x = (unsigned long long)first + (((unsigned long long)b << 32) / end_inv);
            lo = 0; hi = ws.n;
            while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if ((unsigned long long)ws.end[mid] > x) hi = mid; else lo = mid + 1; }
            t[WS_NB + 1u + b] = (uint16_t)(b == WS_NB ? ws.n : lo);
        }
        __syncwarp();
    }
    const uint32_t *ss = seg_start + d.seg_off, *se = seg_end + d.seg_off;
    uint64_t *keys = scratch + scratch_off[unit];

    // pass 1: working set, ltotal, largest
    uint32_t nw = 0, lt = 0, largest = 0;
    for (uint32_t b0 = 0; b0 < d.seg_n; b0 += 32) {
        uint32_t i = b0 + lane;
        uint32_t s = 0, e = 0, ov = 0;
        if (i < d.seg_n) { s = ss[i]; e = se[i]; ov = ws_overlap(ws, s, e); }
        bool keep = ov > 0;
        uint32_t m = __ballot_sync(GATB_FULL, keep);
        if (keep) keys[nw + __popc(m & ((1u << lane) - 1))] = (uint64_t)(e - s);
        nw += __popc(m);
        lt += ov;
        largest = max(largest, keep ? (e - s) : 0u);
    }
    lt = __reduce_add_sync(GATB_FULL, lt);
    largest = __reduce_max_sync(GATB_FULL, largest);
    __syncwarp();

    uint32_t bucket = bucket_size, err = 0;
    unsigned long long drawable = 0;        // sum of the table without its last (largest) entry
    if (nw > 0) {
        // nbuckets == 0: no length histogram wanted (SamplerShift never calls getLengthDistribution,
        // gat/Engine.pyx:1060-1062): the table holds the plain lengths and nothing is "too large"
        const bool hist = nbuckets != 0;
        if (!hist) bucket = 1;
        else if (bucket == 0) bucket = (uint32_t)ceil((double)largest / (double)nbuckets);
        // pass 2: bucket index * bucket, then sort
        for (uint32_t i = lane; i < nw; i += 32) {
            uint32_t l = (uint32_t)keys[i];
            int idx = (int)(((double)l + (double)bucket - 1.0) / (double)bucket);
            if (hist && idx >= (int)nbuckets) err = 1;
            keys[i] = (uint64_t)((uint32_t)idx * bucket);
        }
        err = __any_sync(GATB_FULL, err) ? 1u : 0u;
        uint32_t N = next_pow2(nw);
        for (uint32_t i = nw + lane; i < N; i += 32) keys[i] = GATB_KEY_INF;
        __syncwarp();
        warp_bitonic_sort(keys, N);
        for (uint32_t i = lane; i < nw; i += 32) {
            len_tab[d.tab_off + i] = (uint32_t)keys[i];
            if (i + 1u < nw || nw == 1u) drawable += keys[i];
        }
        drawable = __reduce_add_sync(GATB_FULL, (uint32_t)drawable) + ((unsigned long long)__reduce_add_sync(GATB_FULL, (uint32_t)(drawable >> 32)) << 32);
    }
    if (lane == 0) {
        d.tab_n = nw;
        d.bucket = bucket ? bucket : 1u;
        d.ltotal = (int32_t)lt;
        // Buffer capacity: twice the working segments (room for the counting sort's scratch) and, for skewed
        // units, the expected number of placements -- HistogramSampler draws ranks 1 .. n-1 only
        // (gat/Engine.pyx:420), so a unit whose largest segment holds most of the bases is refilled with the
        // smaller lengths and needs far more placements than it has segments.  An estimate: a unit that still
        // outgrows its buffer is reported (UNIT_OVERFLOW) and the host grows it and runs the call again.
        uint64_t est = 0;
        if (nw > 0) {
            const uint64_t ndraw = nw > 1u ? nw - 1u : 1u;
            const uint64_t mean = drawable / ndraw > 0 ? drawable / ndraw : 1u;
            est = (uint64_t)lt / mean;
            est = est + est / 4u + 64u;
            if (est > (1u << 24)) est = 1u << 24;
        }
        d.cap = next_pow2(max(max(2u * nw + 64u, d.seg_n), (uint32_t)est));   // SamplerSegments places seg_n segments
        d.error = err;
        // the counting sort's bucket plan: every placement starts in [first workspace start - longest length, last
        // workspace end), and about as many placements as working segments are expected
        d.plan_lo = d.plan_inv = d.plan_nb = 0;
        if (nw > 0) {
            const uint32_t lmax = (uint32_t)keys[nw - 1u] + d.bucket, w0 = ws.start[0];   // (the sorted table's last entry)
            const SortPlan pl = make_sort_plan(nw, w0 > lmax ? w0 - lmax : 0u, ws.end[ws.n - 1u]);
            d.plan_lo = pl.lo; d.plan_inv = pl.inv; d.plan_nb = pl.nb;
        }
        units[unit] = d;
    }
}

void launch_prep_units(cudaStream_t st, UnitDesc *units, uint32_t n_units,
                       const uint32_t *seg_start, const uint32_t *seg_end,
                       const uint32_t *ws_start, const uint32_t *ws_end, const uint32_t *ws_cuminc,
                       uint32_t *len_tab, uint64_t *scratch, const uint64_t *scratch_off,
                       uint32_t bucket_size, uint32_t nbuckets, uint32_t *ws_tab)
{
    if (n_units == 0) return;
    const int warps_per_block = 4;
    unsigned blocks = (n_units + warps_per_block - 1) / warps_per_block;
    prep_units_kernel<<<blocks, warps_per_block * 32, 0, st>>>(units, n_units, seg_start, seg_end, ws_start,
                                                                ws_end, ws_cuminc, len_tab, scratch, scratch_off,
                                                                bucket_size, nbuckets, ws_tab);
}

}  // namespace gatb
