// ptx.cuh -- the inline-PTX accessors of the kernels (sm_100a).  Counting kernel: shared memory by 32-bit shared
// address, read-only vector loads by 64-bit global address, a clamping shift and the accumulator address as one IMAD.
// Statistics: TMA bulk copies global -> shared with mbarrier completion.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace gatb {

// shared-memory accesses by 32-bit shared address (the base is computed once, not per access)
__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint4 lds128(uint32_t addr)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t addr)
{
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t lds32(uint32_t addr)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint4 v)
{
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void sts32(uint32_t addr, uint32_t v)
{
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ void red_add_shared(uint32_t addr, uint32_t v)
{
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
// read-only 8-byte global load by 64-bit global address
__device__ __forceinline__ uint2 ldg_nc_u2(uint64_t addr)
{
    uint2 v;
    asm("ld.global.nc.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(addr));
    return v;
}
// read-only 16-byte global load (address 16-byte aligned)
__device__ __forceinline__ uint4 ldg_nc_u4(uint64_t addr)
{
    uint4 v;
    asm("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(addr));
    return v;
}
// v << n, 0 for n >= 32 (PTX shl clamps the shift amount, C++ << does not)
__device__ __forceinline__ uint32_t shl_clamp(uint32_t v, uint32_t n)
{
    uint32_t r;
    asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(v), "r"(n));
    return r;
}
// cell of track (wy & 0xfff) in the accumulators at shared address acc_addr
__device__ __forceinline__ uint32_t acc_cell(uint32_t wy, uint32_t acc_addr)
{
    uint32_t cell;
    asm("mad.lo.u32 %0, %1, 4, %2;" : "=r"(cell) : "r"(wy & 0xfffu), "r"(acc_addr));
    return cell;
}

// ---- TMA bulk copy global -> shared, completion counted in bytes on an mbarrier (shared addresses as above) ----
__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t arrivals)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(arrivals) : "memory");
}
// makes the initialised barriers visible to the async proxy (the TMA unit) before the first copy names them
__device__ __forceinline__ void fence_mbar_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// the one arrival of a phase, announcing `bytes` of copies that will complete on the barrier
__device__ __forceinline__ void mbar_expect_tx(uint32_t mbar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
// dst (shared), src (global) 16-byte aligned, bytes a multiple of 16
__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t mbar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(mbar) : "memory");
}
// true once the phase of the given parity has completed (the data of its copies is then visible to the caller)
__device__ __forceinline__ bool mbar_try_wait(uint32_t mbar, uint32_t parity)
{
    uint32_t done;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done) : "r"(mbar), "r"(parity) : "memory");
    return done != 0u;
}

// ---- 96-bit integer accumulation on the carry chain ----
// (hi:lo) += v * v   (2^32 terms of < 2^64 each fit 96 bits); ptxas turns this into IMAD.WIDE.U32 with a carry-out
// and one add-with-carry
__device__ __forceinline__ void add96_sq(unsigned long long &lo, uint32_t &hi, uint32_t v)
{
    asm("{\n\t.reg .u64 t;\n\tmul.wide.u32 t, %2, %2;\n\tadd.cc.u64 %0, %0, t;\n\taddc.u32 %1, %1, 0;\n\t}"
        : "+l"(lo), "+r"(hi) : "r"(v));
}
// n += carry out of a + b (two instructions, no predicate or select): with b = 2^32 - t this counts a >= t (t >= 1),
// with b = ~t it counts a > t
__device__ __forceinline__ void count_carry(uint32_t &n, uint32_t a, uint32_t b)
{
    asm("{\n\t.reg .u32 t;\n\tadd.cc.u32 t, %1, %2;\n\taddc.u32 %0, %0, 0;\n\t}" : "+r"(n) : "r"(a), "r"(b));
}

}  // namespace gatb
