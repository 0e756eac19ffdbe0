// cp_async.cuh -- thin wrappers over the asynchronous global->shared copy instructions (LDGSTS) used to stage
// per-tile instance lists, and over the vectorised global reductions.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#if defined(SAGARS_CUDA_EMU)
// CPU execution shim of the test suite (tests/cuda_emu/): the same entry points with the instructions' semantics restated on
// the host -- copies land as LATE as the programming model allows, so a read before the matching wait shows up as a failure.
#include "cp_async_emu.h"
#else

namespace sagars {

__device__ __forceinline__ uint32_t smem_u32(const void* p)
{
    return (uint32_t)__cvta_generic_to_shared(p);
}

// 16-byte asynchronous copy, L2 only (streaming data: each row is used by one CTA)
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
// 4-byte asynchronous copy (list entries prefetched many chunks ahead)
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gmem_src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group()
{
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}

// vectorised fire-and-forget global reductions (sm_90+): one instruction adds 4 / 2 floats
__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d)
{
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};\n" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void red_add_v2(float* addr, float a, float b)
{
    asm volatile("red.global.add.v2.f32 [%0], {%1, %2};\n" ::"l"(addr), "f"(a), "f"(b) : "memory");
}
__device__ __forceinline__ void red_add(float* addr, float a)
{
    asm volatile("red.global.add.f32 [%0], %1;\n" ::"l"(addr), "f"(a) : "memory");
}

}  // namespace sagars

#endif  // SAGARS_CUDA_EMU
