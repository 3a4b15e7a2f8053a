// Minimal sm_100a TMA / mbarrier wrappers (inline PTX) used by the tile kernels.
//   loads  : cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes   (SASS UTMALDG)
//   stores : cp.async.bulk.tensor.3d.global.shared::cta.bulk_group                          (SASS UTMASTG)
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace mgw {
namespace tma {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}

// make the barrier init visible to the async proxy before a TMA targets it
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

// generic-proxy smem writes -> visible to the async proxy (before a TMA store reads them)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}

// plain arrival (release): a consumer warp hands a pipeline stage back to the producer
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// named barrier among the first `count` threads' warps of a role (barrier 0 is __syncthreads)
template <int ID, int COUNT>
__device__ __forceinline__ void named_bar_sync()
{
    asm volatile("bar.sync %0, %1;" ::"n"(ID), "n"(COUNT) : "memory");
}

__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "MGW_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra MGW_DONE_%=;\n\t"
        "bra MGW_WAIT_%=;\n\t"
        "MGW_DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

// the same with a suspend-time hint (ns): a waiter that expects to wait long (the producer on `empty`) sleeps in hardware
// instead of spinning through issue slots its SM sub-partition's other warps could use
__device__ __forceinline__ void mbar_wait_hint(uint64_t* bar, uint32_t parity, uint32_t ns)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "MGW_WAITH_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra MGW_DONEH_%=;\n\t"
        "bra MGW_WAITH_%=;\n\t"
        "MGW_DONEH_%=:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity), "r"(ns) : "memory");
}

__device__ __forceinline__ void load_3d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}

__device__ __forceinline__ void store_3d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2)
{
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
                 ::"l"(map), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}

__device__ __forceinline__ void commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// smem sources may be reused / the CTA may exit once the bulk operations have READ them
__device__ __forceinline__ void wait_group_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

// coalesced 16-byte fp32 reduction into global memory (SASS RED.E.ADD.F32x4 ... no return value)
__device__ __forceinline__ void red_add_v4(float* dst, float a, float b, float c, float d)
{
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

__device__ __forceinline__ void prefetch_map(const CUtensorMap* map)
{
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

}  // namespace tma
}  // namespace mgw
