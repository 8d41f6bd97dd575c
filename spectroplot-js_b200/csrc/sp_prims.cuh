// sp_prims.cuh — asynchronous-copy / mbarrier / store primitives shared by the fused kernels (sm_100a PTX):
// mbarrier init / wait / arrive, the 1-D TMA bulk copy global -> shared (SASS UBLKCP) that stages raw frames,
// 256-bit global stores and the shared-memory histogram increment.
#pragma once
#include "sp_kernels.cuh"
#include <cuda.h>          // CUtensorMap (type only: the encoder is resolved through cudaGetDriverEntryPoint)

namespace sp {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// one thread: arm the barrier with the byte count and start the bulk copy global -> shared
__device__ __forceinline__ void tma_load_1d(void *dst_smem, const void *src_gmem, unsigned bytes, uint64_t *bar)
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");       // earlier generic reads of dst vs the async write
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void st_global_256(void *p, uint4 a, uint4 b)
{
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w),
                 "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w) : "memory");
}
__device__ __forceinline__ void red_shared_inc_addr(unsigned addr)
{
    asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(addr) : "memory");
}


// 2-D tensor TMA store shared -> global (SASS UTMASTG): the box shape and the swizzle live in the tensor map
__device__ __forceinline__ void tma_store_2d(const void *tmap, unsigned smem_src, int x, int y)
{
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(tmap), "r"(smem_src), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// the executing thread's bulk groups have finished READING shared memory (the tile may be rewritten)
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// generic-proxy shared-memory writes before this fence are visible to the async proxy (TMA) after it
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

} // namespace sp
