// tests/emu/include/ptx.cuh -- TEST INFRASTRUCTURE: what gat_b200/csrc/ptx.cuh does with inline PTX, in plain C++ for
// the SIMT emulation (tests/emu/include/cuda_runtime.h).  The emulated build of count.cu finds this file first.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

namespace gatb {

__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
template <class T> __device__ __forceinline__ T emu_lds(uint32_t addr) { T v; memcpy(&v, gatb_emu::shared_ptr(addr), sizeof(T)); return v; }
template <class T> __device__ __forceinline__ void emu_sts(uint32_t addr, T v) { memcpy(gatb_emu::shared_ptr(addr), &v, sizeof(T)); }
__device__ __forceinline__ uint4 lds128(uint32_t addr) { return emu_lds<uint4>(addr); }
__device__ __forceinline__ uint2 lds64(uint32_t addr) { return emu_lds<uint2>(addr); }
__device__ __forceinline__ uint32_t lds32(uint32_t addr) { return emu_lds<uint32_t>(addr); }
__device__ __forceinline__ void sts128(uint32_t addr, uint4 v) { emu_sts(addr, v); }
__device__ __forceinline__ void sts32(uint32_t addr, uint32_t v) { emu_sts(addr, v); }
__device__ __forceinline__ void red_add_shared(uint32_t addr, uint32_t v) { emu_sts(addr, emu_lds<uint32_t>(addr) + v); }
__device__ __forceinline__ uint2 ldg_nc_u2(uint64_t addr) { uint2 v; memcpy(&v, (const void *)addr, sizeof(v)); return v; }
__device__ __forceinline__ uint4 ldg_nc_u4(uint64_t addr) { uint4 v; memcpy(&v, (const void *)addr, sizeof(v)); return v; }
__device__ __forceinline__ uint32_t shl_clamp(uint32_t v, uint32_t n) { return n >= 32u ? 0u : v << n; }
__device__ __forceinline__ uint32_t acc_cell(uint32_t wy, uint32_t acc_addr) { return (wy & 0xfffu) * 4u + acc_addr; }

// mbarrier + TMA bulk copy: the copy happens at once, the barrier word counts completed phases
__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t) { emu_sts<uint64_t>(mbar, 0ull); }
__device__ __forceinline__ void fence_mbar_init() {}
__device__ __forceinline__ void mbar_expect_tx(uint32_t, uint32_t) {}
__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t mbar)
{
    if (((uintptr_t)src & 15u) || (dst & 15u) || (bytes & 15u)) { fprintf(stderr, "gatb_emu: misaligned bulk copy\n"); abort(); }
    memcpy(gatb_emu::shared_ptr(dst), src, bytes);
    emu_sts<uint64_t>(mbar, emu_lds<uint64_t>(mbar) + 1ull);
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t mbar, uint32_t parity)
{
    // phases 0 .. n-1 have completed: the phase of parity P is done iff the running phase n has the other parity
    if ((emu_lds<uint64_t>(mbar) & 1ull) != (uint64_t)parity) return true;
    gatb_emu::yield();
    return false;
}

__device__ __forceinline__ void add96_sq(unsigned long long &lo, uint32_t &hi, uint32_t v)
{
    const unsigned long long t = (unsigned long long)v * v;
    lo += t;
    hi += (lo < t) ? 1u : 0u;
}

__device__ __forceinline__ void count_carry(uint32_t &n, uint32_t a, uint32_t b) { n += (uint32_t)(((uint64_t)a + b) >> 32); }

}  // namespace gatb
