// place.cuh -- placement kernels (K1/K2) and the sample-invariant unit preparation.
//
// Replaces SamplerAnnotator.sample (gat/Engine.pyx:515-646) with its helpers HistogramSampler
// (:387-440), SegmentListSampler (:245-353), SegmentList.merge/intersect/filter/trim_ends
// (gat/SegmentList.pyx) and IntervalDictionary.fromIsochores (gat/Engine.pyx:2857-2876).
#pragma once

#include "common.cuh"

namespace gatb {

// status bits per (sample, unit)
enum { UNIT_HIT_ROUND_CAP = 1, UNIT_OVERFLOW = 2 };

// One placement unit = one key ("contig" or "contig.isochore") of one segment track.
struct UnitDesc {
    uint32_t ws_off;      // first workspace piece (into ws_start/ws_end/ws_cuminc)
    uint32_t ws_n;        // number of workspace pieces
    uint32_t ws_total;    // total workspace bases of the unit
    uint32_t seg_off;     // raw segments of the unit (into seg arrays)
    uint32_t seg_n;
    uint32_t tab_off;     // length table: sorted (bucket index * bucket) of the working segments
    uint32_t tab_n;       // = number of working segments (HistogramSampler.total_size)
    uint32_t bucket;      // bucket size actually used
    int32_t  ltotal;      // bases to reproduce (gat/Engine.pyx:550-552)
    uint32_t cap;         // power-of-two capacity of the unit's working buffer
    uint32_t contig;      // contig index
    uint32_t error;       // GATB_ERR_TOO_LARGE etc. from preparation
    uint64_t buf_off;     // offset of the working buffer inside one sample's region
    uint32_t ws_tab_off;  // the unit's bucket tables in PlaceParams.ws_tab (32-bit words; common.cuh), 0xffffffff: none
    uint32_t plan_lo, plan_inv, plan_nb;   // counting-sort plan of the unit's first checkpoint (common.cuh SortPlan)
};

struct PlaceParams {
    const UnitDesc *units;
    const uint32_t *order;       // unit ids, heaviest first
    const uint32_t *ws_start, *ws_end, *ws_cuminc;
    const uint32_t *len_tab;
    const uint32_t *ws_tab;      // bucket tables of the units that have them (WsView::tabw)
    uint64_t *buf;               // [n_samples][sample_stride] packed segments
    uint64_t sample_stride;
    uint32_t *out_n;             // [n_samples][out_n_stride]: per unit (isochores) or per contig
    uint32_t out_n_stride;
    int out_by_contig;           // 1: index out_n by contig (no isochores), 0: by unit
    uint8_t *status;             // [n_samples][n_units]
    uint32_t *unit_over;         // [n_units]: set when any sample of the unit overflowed its buffer (the caller
                                 // grows those units and runs the call again)
    uint32_t n_units;
    int one_piece;               // 1: every unit's workspace is one piece (place_kernel<true>)
    uint32_t n_samples;          // samples in this launch
    uint64_t sample_begin;       // global index of the first sample
    PhiloxKeys keys;             // round keys of the 64-bit seed (philox_keys)
    uint32_t track;
    int sampler_kind;            // 0: SamplerAnnotator (gat/Engine.pyx:445-646), 1: SamplerSegments (:653-737),
                                 // 2: SamplerShift (:998-1111, shift_kernel)
    const uint32_t *seg_start, *seg_end;   // raw segments of the units (UnitDesc.seg_off / seg_n); kind 2 only
    double shift_half_radius;    // SamplerShift: radius / 2 (:1054)
    int32_t shift_extension;     // SamplerShift: extension (0 = use the radius, :1074-1077)
};

struct MergeParams {             // K2: per (sample, contig) concat + merge(0) of the contig's units
    const UnitDesc *units;
    const uint32_t *contig_unit_off;   // [n_contigs+1]
    const uint32_t *contig_units;      // unit ids grouped by contig, in unit order
    const uint64_t *contig_base;       // [n_contigs] offset inside one sample's contig-level region
    const uint64_t *unit_buf;          // [n_samples][unit_stride]
    uint64_t unit_stride;
    const uint32_t *unit_n;            // [n_samples][n_units]
    uint64_t *placed;                  // [n_samples][placed_stride]
    uint64_t placed_stride;
    uint32_t *placed_n;                // [n_samples][n_contigs]
    uint32_t n_units, n_contigs, n_samples;
};

void launch_prep_units(cudaStream_t st, UnitDesc *units, uint32_t n_units,
                       const uint32_t *seg_start, const uint32_t *seg_end,
                       const uint32_t *ws_start, const uint32_t *ws_end, const uint32_t *ws_cuminc,
                       uint32_t *len_tab, uint64_t *scratch, const uint64_t *scratch_off,
                       uint32_t bucket_size, uint32_t nbuckets, uint32_t *ws_tab);
void launch_place(cudaStream_t st, const PlaceParams &p);
void launch_contig_merge(cudaStream_t st, const MergeParams &p);

}  // namespace gatb
