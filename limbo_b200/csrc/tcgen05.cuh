// limbo_b200/csrc/tcgen05.cuh — shared pieces of the TMA + tcgen05 + TMEM kernels (tf32_query.cu, query_i8.cu):
// bounded mbarrier waits that raise an error flag instead of hanging, 2-D TMA loads, MMA commits, TMEM loads and the
// driver's tensor-map encoder.
#pragma once
#include "common.cuh"
#include <cuda.h>

namespace lbtc {

constexpr long long SPIN_LIMIT = 1LL << 24;

__device__ __forceinline__ void mbar_init(uint64_t* b, uint32_t n)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(lb_smem_u32(b)), "r"(n));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* b, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(lb_smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* b)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(lb_smem_u32(b)) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint64_t* b, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(lb_smem_u32(b)), "r"(parity)
        : "memory");
    return ok != 0;
}
// bounded wait: returns false (and raises *err) instead of spinning forever
// The error flag (global memory) is polled only every 1024 attempts: a volatile load per spin from six spinning warps
// would saturate the SM's load/store path (and starve any kernel sharing the SM).
__device__ __forceinline__ bool mbar_wait(uint64_t* b, uint32_t parity, int* err)
{
    long long spins = 0;
    while (!mbar_try(b, parity)) {
        if ((++spins & 1023) == 0 && (spins > SPIN_LIMIT || *(volatile int*)err)) {
            atomicExch(err, 1);
            return false;
        }
    }
    return true;
}
// Long waits of a whole warp (epilogue waiting for ~100 us of MMAs): one lane polls with a back-off, the other 31 lanes
// sleep at the warp barrier instead of issuing try_wait / branch instructions.
__device__ __forceinline__ bool mbar_wait_warp(uint64_t* b, uint32_t parity, int* err)
{
    int ok = 1;
    if ((threadIdx.x & 31) == 0) {
        long long spins = 0;
        while (!mbar_try(b, parity)) {
            __nanosleep(128);
            if ((++spins & 255) == 0 && (spins > (SPIN_LIMIT >> 4) || *(volatile int*)err)) {
                atomicExch(err, 1);
                ok = 0;
                break;
            }
        }
    }
    ok = __shfl_sync(0xffffffffu, ok, 0);
    return ok != 0;
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                     lb_smem_u32(dst)),
                 "l"(map), "r"(c0), "r"(c1), "r"(lb_smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(lb_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn get_encode()
{
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

} // namespace lbtc
