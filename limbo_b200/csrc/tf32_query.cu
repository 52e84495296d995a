// limbo_b200/csrc/tf32_query.cu — reduced-precision candidate scoring on the 5th-generation tensor cores
// (BASELINE.json config 4: N = 16384, D = 12, 1M EI candidates; LB_PREC_TF32 / LB_PREC_FP16).
//
// The per-candidate variance needs |L^-1 k*|^2, i.e. V = L^-1 K* (M N^2 flops, gp.hpp:618-624 once per
// candidate in the reference).  fp64 has no tcgen05 kind, so the fp64 path runs on DMMA (query.cu).  Here the
// factor is inverted once in fp64 (lml.cu, recursive trtri), cast to a row-major tf32 (fp32 container) or fp16 copy, and
//     D[c, n] = sum_{k <= n} Kt[c, k] * Linv[n, k]          (Kt = K*^T, candidates x training points)
// runs on tcgen05.mma with fp32 accumulators in TMEM; the epilogue never writes D: each of the 128 epilogue threads of a
// CTA owns one candidate (one TMEM lane) and accumulates sum_n D[c, n]^2.
//
// Kernels (all persistent, 192 threads: warp 0 = TMA producer, warp 1 = TMEM allocator + single-thread MMA issuer,
// warps 2..5 = epilogue; 4-stage shared-memory ring of 128-byte SWIZZLE_128B rows; every mbarrier wait is bounded and
// raises an error flag instead of hanging the GPU):
//   pair_gemm_norm_kernel          DEFAULT.  Two CTAs = one MMA pair (tcgen05 ... cta_group::2, UMMA M = 256): each CTA
//                                  owns 128 candidates and half of every B tile; each A slab feeds two n-tiles (all 512
//                                  TMEM columns).  24 KB from L2 per 128x256x64-MAC unit instead of 40 KB.
//   tf32_gemm_norm_cluster_kernel  fallback (LB_TF32_PAIR=0): clusters of 2 / 4 CTAs share the candidate tile by TMA
//                                  multicast, split the n-tiles, double-buffered accumulators.
//   tf32_gemm_norm_kernel          single CTA, 128 x 256 tiles (LB_TF32_CLUSTER=1; also the validation entry that can
//                                  write D).
// Around them: kstar_t32_kernel (K*^T chunk from fp64 kernel evaluations with the squared distances on the fp64 tensor pipe,
// mean and rounding-bias partials fused), mu_reduce_kernel, sigma2_t32_kernel (clamp / noise of gp.hpp:623,166 and the
// rounding-bias correction), linv_to_rowmajor_kernel (+ absmax / colnorm2 for the fp16 scale and the bias weights).
#include "tcgen05.cuh"
#include <cuda_fp16.h>
#include <cmath>
#include <type_traits>
#include <cstdlib>

namespace tf32q {

using namespace lbtc;

constexpr int BM = 128;       // candidates per tile (UMMA M)
constexpr int BN = 256;       // outputs (rows of L^-1) per tile (UMMA N)
// k elements per stage = 128 B = one swizzle atom row: 32 tf32 or 64 fp16; one stage is always 4 MMAs (K = 8 tf32 / 16 fp16)
template <bool F16> __host__ __device__ constexpr int bke() { return F16 ? 64 : 32; }
constexpr int MMAS_PER_STAGE = 4;
constexpr int STAGES = 4;
constexpr int A_BYTES = BM * 128;  // 16 KB
constexpr int B_BYTES = BN * 128;  // 32 KB
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int THREADS = 192;
constexpr size_t SMEM_BYTES = (size_t)STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;
// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor, mma_sm100_desc.hpp):
//   [0,14) start address >> 4 | [16,30) leading byte offset >> 4 (unused for swizzled K-major: 1) |
//   [32,46) stride byte offset >> 4 (8 rows x 128 B = 1024 B -> 64) | [46,48) version = 1 | [61,64) layout = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr)
{
    return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32 = 1 @4, a/b format TF32 = 2 @7/@10,
// a/b K-major (0) @15/@16, N >> 3 @17, M >> 4 @24
// a/b format: F16 = 0, TF32 = 2
template <bool F16>
__host__ __device__ constexpr uint32_t idesc()
{
    return (1u << 4) | ((F16 ? 0u : 2u) << 7) | ((F16 ? 0u : 2u) << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}

template <bool F16>
__device__ __forceinline__ void umma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t accumulate)
{
    if (F16)
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc<true>()), "r"(accumulate)
            : "memory");
    else
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc<false>()), "r"(accumulate)
            : "memory");
}
// D[c, n] = sum_k A[c, k] B[n, k]; tri != 0: k only up to the end of the n-tile (B lower triangular).
// norm2[c] += sum_n D[c, n]^2 ; Dout (optional, row-major M x N) receives D for validation.
template <bool F16>
__global__ void __launch_bounds__(THREADS, 1)
tf32_gemm_norm_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, int64_t M, int64_t N,
    int64_t K, int tri, float* __restrict__ norm2, float* __restrict__ Dout, int* __restrict__ err)
{
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023); // SWIZZLE_128B needs 1024-byte alignment
    uint64_t* full = (uint64_t*)(smem + (size_t)STAGES * STAGE_BYTES);
    uint64_t* empty = full + STAGES;
    uint64_t* tfull = empty + STAGES;   // [2]
    uint64_t* tempty = tfull + 2;       // [2]
    uint32_t* tmem_base_s = (uint32_t*)(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m_tiles = (int)(M / BM), n_tiles = (int)(N / BN);

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) { // TMEM: 512 columns (2 accumulators of 256)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(lb_smem_u32(tmem_base_s)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_base_s;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            int s = 0; uint32_t ph = 0; bool ok = true;
            for (int mt = blockIdx.x; mt < m_tiles && ok; mt += gridDim.x) {
                for (int nt = 0; nt < n_tiles && ok; ++nt) {
                    const int64_t kend = tri ? (int64_t)(nt + 1) * BN : K;
                    const int kblocks = (int)((kend < K ? kend : K) / bke<F16>());
                    for (int kb = 0; kb < kblocks; ++kb) {
                        if (!mbar_wait(&empty[s], ph ^ 1, err)) { ok = false; break; }
                        uint8_t* sa = smem + (size_t)s * STAGE_BYTES;
                        mbar_expect_tx(&full[s], STAGE_BYTES);
                        tma_load_2d(sa, &mapA, kb * bke<F16>(), mt * BM, &full[s]);
                        tma_load_2d(sa + A_BYTES, &mapB, kb * bke<F16>(), nt * BN, &full[s]);
                        if (++s == STAGES) { s = 0; ph ^= 1; }
                    }
                }
            }
        }
    }
    else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            int s = 0; uint32_t ph = 0; bool ok = true;
            int buf = 0; uint32_t tph[2] = {0, 0};
            for (int mt = blockIdx.x; mt < m_tiles && ok; mt += gridDim.x) {
                for (int nt = 0; nt < n_tiles && ok; ++nt) {
                    const int64_t kend = tri ? (int64_t)(nt + 1) * BN : K;
                    const int kblocks = (int)((kend < K ? kend : K) / bke<F16>());
                    if (!mbar_wait(&tempty[buf], tph[buf] ^ 1, err)) { ok = false; break; } // epilogue drained this accumulator
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t d_tmem = tmem_base + (uint32_t)(buf * BN);
                    for (int kb = 0; kb < kblocks; ++kb) {
                        if (!mbar_wait(&full[s], ph, err)) { ok = false; break; }
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        const uint32_t sa = lb_smem_u32(smem + (size_t)s * STAGE_BYTES);
                        const uint64_t adesc = make_desc(sa), bdesc = make_desc(sa + A_BYTES);
#pragma unroll
                        for (int k = 0; k < MMAS_PER_STAGE; ++k) // +32 B per MMA inside the 128 B swizzle row: +2 in the >>4 address field
                            umma<F16>(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), (kb | k) != 0);
                        umma_commit(&empty[s]); // frees the smem slot when these MMAs have read it
                        if (++s == STAGES) { s = 0; ph ^= 1; }
                    }
                    umma_commit(&tfull[buf]); // accumulator complete
                    tph[buf] ^= 1;
                    buf ^= 1;
                }
            }
        }
    }
    else {
        // ===== epilogue: warps 2..5, TMEM lane quarter = warp % 4 =====
        const int q = warp & 3;
        const int row = q * 32 + lane; // candidate inside the tile == TMEM lane
        int buf = 0; uint32_t tph[2] = {0, 0}; bool ok = true;
        for (int mt = blockIdx.x; mt < m_tiles && ok; mt += gridDim.x) {
            float acc = 0.f;
            for (int nt = 0; nt < n_tiles && ok; ++nt) {
                if (!mbar_wait_warp(&tfull[buf], tph[buf], err)) { ok = false; break; }
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN);
#pragma unroll 1
                for (int c = 0; c < BN; c += 32) {
                    uint32_t v[32];
                    tmem_ld32(taddr + c, v);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float d = __uint_as_float(v[j]);
                        acc = fmaf(d, d, acc);
                        if (Dout) Dout[((int64_t)mt * BM + row) * N + (int64_t)nt * BN + c + j] = d;
                    }
                }
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty[buf]); // 4 arrivals (one per epilogue warp) release the accumulator
                tph[buf] ^= 1;
                buf ^= 1;
            }
            if (ok) norm2[(int64_t)mt * BM + row] = acc;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------
// Clustered variant: CL CTAs (CL = 2 or 4) share one candidate tile and split the n-tiles between them.  The A
// tile (K*^T, private to a candidate tile, streamed from HBM once per n-tile) is loaded ONCE per cluster and
// TMA-multicast into every CTA's shared memory, which divides the dominant HBM stream by CL; each CTA keeps its own
// B tiles, TMEM accumulators, MMA issuer and epilogue.  Slot reuse is cluster-wide: every MMA commit multicasts its
// "slot free" arrival to all CTAs of the cluster (empty barriers count CL arrivals).
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d_mcast(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar, uint16_t mask)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%2, %3}], [%4], %5;"
        ::"r"(lb_smem_u32(dst)), "l"(map), "r"(c0), "r"(c1), "r"(lb_smem_u32(bar)), "h"(mask)
        : "memory");
}
__device__ __forceinline__ void umma_commit_mcast(uint64_t* bar, uint16_t mask)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                     lb_smem_u32(bar)),
                 "h"(mask)
                 : "memory");
}

// norm2 is [CL][M]: each CTA of a cluster writes the partial sum over its own n-tiles (summed later, fixed order).
template <int CL, bool F16>
__global__ void __launch_bounds__(THREADS, 1)
tf32_gemm_norm_cluster_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, int64_t M, int64_t N,
    int64_t K, int tri, float* __restrict__ norm2, int* __restrict__ err)
{
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* full = (uint64_t*)(smem + (size_t)STAGES * STAGE_BYTES);
    uint64_t* empty = full + STAGES;
    uint64_t* tfull = empty + STAGES;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_base_s = (uint32_t*)(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rank = (int)cluster_ctarank();
    const int cluster_id = blockIdx.x / CL, nclusters = gridDim.x / CL;
    const int m_tiles = (int)(M / BM), n_groups = (int)(N / BN) / CL; // N is a multiple of BN * CL
    constexpr uint16_t ALL = (uint16_t)((1u << CL) - 1);

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], CL); }
        for (int b = 0; b < 2; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(lb_smem_u32(tmem_base_s)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    cluster_sync_all(); // every CTA's barriers are initialised before any remote arrival / multicast can target them
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_base_s;

    if (warp == 0) {
        if (lane == 0) { // ===== TMA producer: own B tile; rank 0 additionally multicasts the shared A tile =====
            int s = 0; uint32_t ph = 0; bool ok = true;
            for (int mt = cluster_id; mt < m_tiles && ok; mt += nclusters) {
                for (int grp = 0; grp < n_groups && ok; ++grp) {
                    const int nt = grp * CL + rank;
                    const int64_t kend = tri ? (int64_t)(grp + 1) * CL * BN : K; // the whole cluster walks the same k range
                    const int kblocks = (int)((kend < K ? kend : K) / bke<F16>());
                    for (int kb = 0; kb < kblocks; ++kb) {
                        if (!mbar_wait(&empty[s], ph ^ 1, err)) { ok = false; break; } // freed by ALL CTAs of the cluster
                        uint8_t* sa = smem + (size_t)s * STAGE_BYTES;
                        mbar_expect_tx(&full[s], STAGE_BYTES);
                        if (rank == 0) tma_load_2d_mcast(sa, &mapA, kb * bke<F16>(), mt * BM, &full[s], ALL);
                        tma_load_2d(sa + A_BYTES, &mapB, kb * bke<F16>(), nt * BN, &full[s]);
                        if (++s == STAGES) { s = 0; ph ^= 1; }
                    }
                }
            }
        }
    }
    else if (warp == 1) {
        if (lane == 0) { // ===== MMA issuer =====
            int s = 0; uint32_t ph = 0; bool ok = true;
            int buf = 0; uint32_t tph[2] = {0, 0};
            for (int mt = cluster_id; mt < m_tiles && ok; mt += nclusters) {
                for (int grp = 0; grp < n_groups && ok; ++grp) {
                    const int64_t kend = tri ? (int64_t)(grp + 1) * CL * BN : K;
                    const int kblocks = (int)((kend < K ? kend : K) / bke<F16>());
                    if (!mbar_wait(&tempty[buf], tph[buf] ^ 1, err)) { ok = false; break; }
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t d_tmem = tmem_base + (uint32_t)(buf * BN);
                    for (int kb = 0; kb < kblocks; ++kb) {
                        if (!mbar_wait(&full[s], ph, err)) { ok = false; break; }
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        const uint32_t sa = lb_smem_u32(smem + (size_t)s * STAGE_BYTES);
                        const uint64_t adesc = make_desc(sa), bdesc = make_desc(sa + A_BYTES);
#pragma unroll
                        for (int k = 0; k < MMAS_PER_STAGE; ++k)
                            umma<F16>(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), (kb | k) != 0);
                        umma_commit_mcast(&empty[s], ALL); // this CTA is done with slot s: tell every producer of the cluster
                        if (++s == STAGES) { s = 0; ph ^= 1; }
                    }
                    umma_commit(&tfull[buf]);
                    tph[buf] ^= 1;
                    buf ^= 1;
                }
            }
        }
    }
    else {
        const int q = warp & 3;
        const int row = q * 32 + lane;
        int buf = 0; uint32_t tph[2] = {0, 0}; bool ok = true;
        for (int mt = cluster_id; mt < m_tiles && ok; mt += nclusters) {
            float acc = 0.f;
            for (int grp = 0; grp < n_groups && ok; ++grp) {
                if (!mbar_wait_warp(&tfull[buf], tph[buf], err)) { ok = false; break; }
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN);
#pragma unroll 1
                for (int c = 0; c < BN; c += 32) {
                    uint32_t v[32];
                    tmem_ld32(taddr + c, v);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float d = __uint_as_float(v[j]);
                        acc = fmaf(d, d, acc);
                    }
                }
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty[buf]);
                tph[buf] ^= 1;
                buf ^= 1;
            }
            if (ok) norm2[(int64_t)rank * M + (int64_t)mt * BM + row] = acc;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    cluster_sync_all(); // nobody leaves while a peer may still multicast into its shared memory / barriers
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------
// CTA-pair variant (tcgen05 cta_group::2): the GEMM above is bound by operand delivery from L2 (11.2 TB/s measured at
// 128 x 256 tiles, the LTS cap of the chip is ~12 TB/s), so the lever is bytes per MAC.  Two CTAs of a cluster form one
// MMA pair: UMMA M = 256 (each CTA owns 128 candidates = its own A rows and its own TMEM lanes) and every B tile is split
// between the two CTAs (128 of the 256 rows of L^-1 each), so B is fetched once per 256 candidates.  Each A slab is used
// for TWO n-tiles (two 256-column accumulators = all 512 TMEM columns): per 128 x 256 x 64-MAC unit a CTA pulls
// 8 KB (A) + 16 KB (B) instead of 8 + 32 KB.  Only the leader CTA issues MMAs; both CTAs run a TMA producer whose
// transactions complete on the LEADER's "full" barrier; commits are multicast to both CTAs ("slot free", "accumulators
// full"); both epilogues report "accumulators drained" to the leader.
// ---------------------------------------------------------------------------------------------------------
constexpr int HB_BYTES = (BN / 2) * 128;                    // half of a B tile: 128 rows x 128 B
constexpr int PAIR_STAGE_BYTES = A_BYTES + 2 * HB_BYTES;    // A + B(n0) half + B(n1) half = 48 KB
constexpr size_t PAIR_SMEM_BYTES = (size_t)STAGES * PAIR_STAGE_BYTES + 1024 + 256;

__device__ __forceinline__ uint32_t mapa_u32(uint32_t smem_addr, uint32_t cta)
{
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(cta));
    return r;
}
// TMA load whose bytes complete on a barrier given by its shared::cluster address (the leader's)
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* map, int c0, int c1, uint32_t bar_cluster_addr)
{
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                     lb_smem_u32(dst)),
                 "l"(map), "r"(c0), "r"(c1), "r"(bar_cluster_addr)
                 : "memory");
}
template <bool F16>
__host__ __device__ constexpr uint32_t idesc_pair()
{
    return (1u << 4) | ((F16 ? 0u : 2u) << 7) | ((F16 ? 0u : 2u) << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((2 * BM) >> 4) << 24);
}
template <bool F16>
__device__ __forceinline__ void umma_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t accumulate)
{
    if (F16)
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc_pair<true>()), "r"(accumulate)
            : "memory");
    else
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc_pair<false>()), "r"(accumulate)
            : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar)
{
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(lb_smem_u32(bar)),
                 "h"((uint16_t)3)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_cluster_addr)
{
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster_addr) : "memory");
}

// M % 256 == 0, N % 512 == 0.  norm2[c] = sum_n D[c, n]^2 (one partial per candidate).
template <bool F16>
__global__ void __launch_bounds__(THREADS, 1)
pair_gemm_norm_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, int64_t M, int64_t N, int64_t K,
    int tri, float* __restrict__ norm2, int* __restrict__ err)
{
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* full = (uint64_t*)(smem + (size_t)STAGES * PAIR_STAGE_BYTES);
    uint64_t* empty = full + STAGES;
    uint64_t* tfull = empty + STAGES;
    uint64_t* tempty = tfull + 1;
    uint32_t* tmem_base_s = (uint32_t*)(tempty + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rank = (int)cluster_ctarank();
    const int pair_id = blockIdx.x >> 1, npairs = gridDim.x >> 1;
    const int m_pairs = (int)(M / (2 * BM)), n_groups = (int)(N / (2 * BN));
    constexpr int BKE = bke<F16>();

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(tfull, 1);
        mbar_init(tempty, 8); // 4 epilogue warps of each CTA of the pair (leader's copy is the one waited on)
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) { // the same warp of BOTH CTAs performs the pair-wide allocation (all 512 columns)
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(lb_smem_u32(tmem_base_s)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    cluster_sync_all();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_base_s;

    auto kblocks_of = [&](int nt) {
        const int64_t kend = tri ? (int64_t)(nt + 1) * BN : K;
        return (int)((kend < K ? kend : K) / BKE);
    };

    if (warp == 0) {
        if (lane == 0) { // ===== TMA producer (both CTAs): own A rows, own half of both B tiles; bytes land on the leader's barrier =====
            int s = 0; uint32_t ph = 0; bool ok = true;
            for (int mt = pair_id; mt < m_pairs && ok; mt += npairs) {
                for (int grp = 0; grp < n_groups && ok; ++grp) {
                    const int n0 = 2 * grp, n1 = n0 + 1;
                    const int kb0 = kblocks_of(n0), kb1 = kblocks_of(n1);
                    for (int kb = 0; kb < kb1; ++kb) {
                        if (!mbar_wait(&empty[s], ph ^ 1, err)) { ok = false; break; }
                        const bool has0 = kb < kb0;
                        uint8_t* sa = smem + (size_t)s * PAIR_STAGE_BYTES;
                        const uint32_t lfull = mapa_u32(lb_smem_u32(&full[s]), 0);
                        if (rank == 0) mbar_expect_tx(&full[s], 2u * (uint32_t)(A_BYTES + HB_BYTES + (has0 ? HB_BYTES : 0)));
                        tma_load_2d_pair(sa, &mapA, kb * BKE, mt * 2 * BM + rank * BM, lfull);
                        if (has0) tma_load_2d_pair(sa + A_BYTES, &mapB, kb * BKE, n0 * BN + rank * (BN / 2), lfull);
                        tma_load_2d_pair(sa + A_BYTES + HB_BYTES, &mapB, kb * BKE, n1 * BN + rank * (BN / 2), lfull);
                        if (++s == STAGES) { s = 0; ph ^= 1; }
                    }
                }
            }
        }
    }
    else if (warp == 1) {
        if (lane == 0 && rank == 0) { // ===== MMA issuer: leader CTA only =====
            int s = 0; uint32_t ph = 0; bool ok = true;
            uint32_t tph = 0;
            for (int mt = pair_id; mt < m_pairs && ok; mt += npairs) {
                for (int grp = 0; grp < n_groups && ok; ++grp) {
                    const int kb0 = kblocks_of(2 * grp), kb1 = kblocks_of(2 * grp + 1);
                    if (!mbar_wait(tempty, tph ^ 1, err)) { ok = false; break; }
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    for (int kb = 0; kb < kb1; ++kb) {
                        if (!mbar_wait(&full[s], ph, err)) { ok = false; break; }
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        const uint32_t sa = lb_smem_u32(smem + (size_t)s * PAIR_STAGE_BYTES);
                        const uint64_t adesc = make_desc(sa), b0desc = make_desc(sa + A_BYTES), b1desc = make_desc(sa + A_BYTES + HB_BYTES);
                        if (kb < kb0) {
#pragma unroll
                            for (int k = 0; k < MMAS_PER_STAGE; ++k)
                                umma_pair<F16>(tmem_base, adesc + (uint64_t)(2 * k), b0desc + (uint64_t)(2 * k), (kb | k) != 0);
                        }
#pragma unroll
                        for (int k = 0; k < MMAS_PER_STAGE; ++k)
                            umma_pair<F16>(tmem_base + (uint32_t)BN, adesc + (uint64_t)(2 * k), b1desc + (uint64_t)(2 * k), (kb | k) != 0);
                        umma_commit_pair(&empty[s]); // slot s is free in both CTAs
                        if (++s == STAGES) { s = 0; ph ^= 1; }
                    }
                    umma_commit_pair(tfull); // both accumulators complete, in both CTAs
                    tph ^= 1;
                }
            }
        }
    }
    else { // ===== epilogue (both CTAs): each thread owns one candidate = one TMEM lane of its CTA =====
        const int q = warp & 3;
        const int row = q * 32 + lane;
        const uint32_t ltempty = mapa_u32(lb_smem_u32(tempty), 0);
        uint32_t tph = 0; bool ok = true;
        for (int mt = pair_id; mt < m_pairs && ok; mt += npairs) {
            float acc = 0.f;
            for (int grp = 0; grp < n_groups && ok; ++grp) {
                if (!mbar_wait_warp(tfull, tph, err)) { ok = false; break; }
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
                for (int c = 0; c < 2 * BN; c += 32) {
                    uint32_t v[32];
                    tmem_ld32(taddr + c, v);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float d = __uint_as_float(v[j]);
                        acc = fmaf(d, d, acc);
                    }
                }
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(ltempty);
                tph ^= 1;
            }
            if (ok) norm2[(int64_t)mt * 2 * BM + rank * BM + row] = acc;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    cluster_sync_all(); // neither CTA leaves (or frees TMEM) while the pair may still be using its memory
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------
// Split-operand variant of the CTA-pair kernel (LB_PREC_FP16X3): every operand is carried as hi + 2^-11 lo with hi, lo
// both fp16 (22 significant bits), and
//     D = A_hi B_hi + 2^-11 (A_hi B_lo + A_lo B_hi)            (the 2^-22 A_lo B_lo term is dropped)
// is formed from three fp16 MMAs per k-step into TWO fp32 accumulators (acc0 = hi x hi in TMEM columns [0, 256),
// acc1 = the cross terms in [256, 512)), combined in the epilogue in fp64, where sum_n D^2 is accumulated in fp64 as well.
// One n-tile (256 rows of L^-1) per pass; otherwise the pipeline of pair_gemm_norm_kernel (both CTAs produce, the leader
// issues, commits are multicast).  3x the MMA work and 2x the operand bytes of LB_PREC_FP16 buy |d sigma^2| ~ 1e-6 instead
// of ~2e-3 (tests/test_gpu_config4.py).
// ---------------------------------------------------------------------------------------------------------
constexpr int SPLIT_STAGES = 3;
constexpr int SPLIT_STAGE_BYTES = 2 * A_BYTES + 2 * HB_BYTES; // A_hi, A_lo, B_hi half, B_lo half = 64 KB
constexpr size_t SPLIT_SMEM_BYTES = (size_t)SPLIT_STAGES * SPLIT_STAGE_BYTES + 1024 + 256;

__global__ void __launch_bounds__(THREADS, 1)
pair_split_gemm_norm_kernel(const __grid_constant__ CUtensorMap mapAh, const __grid_constant__ CUtensorMap mapAl,
    const __grid_constant__ CUtensorMap mapBh, const __grid_constant__ CUtensorMap mapBl, int64_t M, int64_t N, int64_t K, int tri,
    double* __restrict__ norm2, int* __restrict__ err)
{
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* full = (uint64_t*)(smem + (size_t)SPLIT_STAGES * SPLIT_STAGE_BYTES);
    uint64_t* empty = full + SPLIT_STAGES;
    uint64_t* tfull = empty + SPLIT_STAGES;
    uint64_t* tempty = tfull + 1;
    uint32_t* tmem_base_s = (uint32_t*)(tempty + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rank = (int)cluster_ctarank();
    const int pair_id = blockIdx.x >> 1, npairs = gridDim.x >> 1;
    const int m_pairs = (int)(M / (2 * BM)), n_tiles = (int)(N / BN);
    constexpr int BKE = bke<true>();

    if (threadIdx.x == 0) {
        for (int s = 0; s < SPLIT_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(tfull, 1);
        mbar_init(tempty, 8);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(lb_smem_u32(tmem_base_s)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    cluster_sync_all();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_base_s;

    auto kblocks_of = [&](int nt) {
        const int64_t kend = tri ? (int64_t)(nt + 1) * BN : K;
        return (int)((kend < K ? kend : K) / BKE);
    };

    if (warp == 0) {
        if (lane == 0) { // ===== TMA producer (both CTAs): own A rows (hi, lo), own half of the B tile (hi, lo) =====
            int s = 0; uint32_t ph = 0; bool ok = true;
            for (int mt = pair_id; mt < m_pairs && ok; mt += npairs) {
                for (int nt = 0; nt < n_tiles && ok; ++nt) {
                    const int kbn = kblocks_of(nt);
                    for (int kb = 0; kb < kbn; ++kb) {
                        if (!mbar_wait(&empty[s], ph ^ 1, err)) { ok = false; break; }
                        uint8_t* sa = smem + (size_t)s * SPLIT_STAGE_BYTES;
                        const uint32_t lfull = mapa_u32(lb_smem_u32(&full[s]), 0);
                        if (rank == 0) mbar_expect_tx(&full[s], 2u * (uint32_t)SPLIT_STAGE_BYTES);
                        tma_load_2d_pair(sa, &mapAh, kb * BKE, mt * 2 * BM + rank * BM, lfull);
                        tma_load_2d_pair(sa + A_BYTES, &mapAl, kb * BKE, mt * 2 * BM + rank * BM, lfull);
                        tma_load_2d_pair(sa + 2 * A_BYTES, &mapBh, kb * BKE, nt * BN + rank * (BN / 2), lfull);
                        tma_load_2d_pair(sa + 2 * A_BYTES + HB_BYTES, &mapBl, kb * BKE, nt * BN + rank * (BN / 2), lfull);
                        if (++s == SPLIT_STAGES) { s = 0; ph ^= 1; }
                    }
                }
            }
        }
    }
    else if (warp == 1) {
        if (lane == 0 && rank == 0) { // ===== MMA issuer: leader CTA only =====
            int s = 0; uint32_t ph = 0; bool ok = true;
            uint32_t tph = 0;
            for (int mt = pair_id; mt < m_pairs && ok; mt += npairs) {
                for (int nt = 0; nt < n_tiles && ok; ++nt) {
                    const int kbn = kblocks_of(nt);
                    if (!mbar_wait(tempty, tph ^ 1, err)) { ok = false; break; }
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    for (int kb = 0; kb < kbn; ++kb) {
                        if (!mbar_wait(&full[s], ph, err)) { ok = false; break; }
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        const uint32_t sa = lb_smem_u32(smem + (size_t)s * SPLIT_STAGE_BYTES);
                        const uint64_t ah = make_desc(sa), al = make_desc(sa + A_BYTES), bh = make_desc(sa + 2 * A_BYTES),
                                       bl = make_desc(sa + 2 * A_BYTES + HB_BYTES);
#pragma unroll
                        for (int k = 0; k < MMAS_PER_STAGE; ++k) umma_pair<true>(tmem_base, ah + (uint64_t)(2 * k), bh + (uint64_t)(2 * k), (kb | k) != 0);
#pragma unroll
                        for (int k = 0; k < MMAS_PER_STAGE; ++k) {
                            umma_pair<true>(tmem_base + (uint32_t)BN, ah + (uint64_t)(2 * k), bl + (uint64_t)(2 * k), (kb | k) != 0);
                            umma_pair<true>(tmem_base + (uint32_t)BN, al + (uint64_t)(2 * k), bh + (uint64_t)(2 * k), 1);
                        }
                        umma_commit_pair(&empty[s]);
                        if (++s == SPLIT_STAGES) { s = 0; ph ^= 1; }
                    }
                    umma_commit_pair(tfull);
                    tph ^= 1;
                }
            }
        }
    }
    else { // ===== epilogue (both CTAs): D = acc0 + 2^-11 acc1 and sum_n D^2, both in fp64 =====
        const int q = warp & 3;
        const int row = q * 32 + lane;
        const uint32_t ltempty = mapa_u32(lb_smem_u32(tempty), 0);
        uint32_t tph = 0; bool ok = true;
        for (int mt = pair_id; mt < m_pairs && ok; mt += npairs) {
            double acc = 0.0;
            for (int nt = 0; nt < n_tiles && ok; ++nt) {
                if (!mbar_wait_warp(tfull, tph, err)) { ok = false; break; }
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
                for (int c = 0; c < BN; c += 32) {
                    uint32_t v0[32], v1[32];
                    tmem_ld32(taddr + c, v0);
                    tmem_ld32(taddr + BN + c, v1);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const double d = fma((double)__uint_as_float(v1[j]), 1.0 / 2048.0, (double)__uint_as_float(v0[j]));
                        acc = fma(d, d, acc);
                    }
                }
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(ltempty);
                tph ^= 1;
            }
            if (ok) norm2[(int64_t)mt * 2 * BM + rank * BM + row] = acc;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    cluster_sync_all();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
    }
}

// row-major (rows x K) fp32 matrix, boxes of 32 k x box_rows rows, 128-byte swizzle, tf32 rounding on load
static int make_map(CUtensorMap* map, const void* base, int64_t rows, int64_t K, int64_t ld, int box_rows, bool f16)
{
    EncodeTiledFn enc = get_encode();
    if (!enc) return LB_ERR_UNSUPPORTED;
    cuuint64_t gdim[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    cuuint64_t gstr[1] = {(cuuint64_t)ld * (f16 ? 2 : 4)};
    cuuint32_t box[2] = {(cuuint32_t)(f16 ? 64 : 32), (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_TFLOAT32, 2, (void*)base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? LB_OK : LB_ERR_CUDA;
}

LbOncePerDevice g_attr_once;

} // namespace tf32q

// A: M x K (ld lda), B: N x K (ld ldb), row-major fp32 (tf32 MMA) or fp16 in device memory; M % 128 == 0, N % 256 == 0, K % 64 == 0.
int lb_launch_tf32_gemm_norm(cudaStream_t st, const void* dA, int64_t lda, const void* dB, int64_t ldb, int64_t M, int64_t N, int64_t K,
    int tri, float* dNorm2, float* dDout, int* dErr, int grid, int f16)
{
    using namespace tf32q;
    if (M % BM || N % BN || K % 64) return LB_ERR_ARG;
    if (g_attr_once.need()) {
        LB_CUDA(cudaFuncSetAttribute(tf32_gemm_norm_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
        LB_CUDA(cudaFuncSetAttribute(tf32_gemm_norm_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
    }
    alignas(64) CUtensorMap mapA, mapB;
    int rc;
    if ((rc = make_map(&mapA, dA, M, K, lda, BM, f16 != 0))) return rc;
    if ((rc = make_map(&mapB, dB, N, K, ldb, BN, f16 != 0))) return rc;
    const int m_tiles = (int)(M / BM);
    if (grid > m_tiles) grid = m_tiles;
    if (f16) tf32_gemm_norm_kernel<true><<<grid, THREADS, SMEM_BYTES, st>>>(mapA, mapB, M, N, K, tri, dNorm2, dDout, dErr);
    else tf32_gemm_norm_kernel<false><<<grid, THREADS, SMEM_BYTES, st>>>(mapA, mapB, M, N, K, tri, dNorm2, dDout, dErr);
    LB_CUDA(cudaGetLastError());
    return LB_OK;
}

// Clustered launch: N must be a multiple of 256 * CL; dNorm2 holds CL partial rows of M floats.
template <int CL, bool F16>
static int launch_cluster(cudaStream_t st, const CUtensorMap& mapA, const CUtensorMap& mapB, int64_t M, int64_t N, int64_t K, int tri,
    float* dNorm2, int* dErr, int grid)
{
    using namespace tf32q;
    static LbOncePerDevice attr_once;
    if (attr_once.need()) {
        LB_CUDA(cudaFuncSetAttribute(tf32_gemm_norm_cluster_kernel<CL, F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(THREADS);
    cfg.dynamicSmemBytes = SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    LB_CUDA(cudaLaunchKernelEx(&cfg, tf32_gemm_norm_cluster_kernel<CL, F16>, mapA, mapB, M, N, K, tri, dNorm2, dErr));
    return LB_OK;
}

int lb_launch_pair_gemm_norm(cudaStream_t st, const void* dA, int64_t lda, const void* dB, int64_t ldb, int64_t M, int64_t N, int64_t K,
    int tri, float* dNorm2, int* dErr, int sms, int f16);
int lb_launch_pair_split_gemm_norm(cudaStream_t st, const void* dAh, const void* dAl, int64_t lda, const void* dBh, const void* dBl, int64_t ldb,
    int64_t M, int64_t N, int64_t K, int tri, double* dNorm2, int* dErr, int sms);

int lb_launch_tf32_gemm_norm_cluster(cudaStream_t st, const void* dA, int64_t lda, const void* dB, int64_t ldb, int64_t M, int64_t N,
    int64_t K, int tri, float* dNorm2, int* dErr, int sms, int cl, int f16)
{
    using namespace tf32q;
    if (M % BM || N % (BN * cl) || K % 64 || (cl != 2 && cl != 4)) return LB_ERR_ARG;
    alignas(64) CUtensorMap mapA, mapB;
    int rc;
    if ((rc = make_map(&mapA, dA, M, K, lda, BM, f16 != 0))) return rc;
    if ((rc = make_map(&mapB, dB, N, K, ldb, BN, f16 != 0))) return rc;
    const int m_tiles = (int)(M / BM);
    int nclusters = sms / cl;
    if (nclusters > m_tiles) nclusters = m_tiles;
    const int grid = nclusters * cl;
    if (f16)
        return cl == 2 ? launch_cluster<2, true>(st, mapA, mapB, M, N, K, tri, dNorm2, dErr, grid)
                       : launch_cluster<4, true>(st, mapA, mapB, M, N, K, tri, dNorm2, dErr, grid);
    return cl == 2 ? launch_cluster<2, false>(st, mapA, mapB, M, N, K, tri, dNorm2, dErr, grid)
                   : launch_cluster<4, false>(st, mapA, mapB, M, N, K, tri, dNorm2, dErr, grid);
}

template <bool F16>
static int launch_pair(cudaStream_t st, const CUtensorMap& mapA, const CUtensorMap& mapB, int64_t M, int64_t N, int64_t K, int tri,
    float* dNorm2, int* dErr, int grid)
{
    using namespace tf32q;
    static LbOncePerDevice attr_once;
    if (attr_once.need()) {
        LB_CUDA(cudaFuncSetAttribute(pair_gemm_norm_kernel<F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PAIR_SMEM_BYTES));
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(THREADS);
    cfg.dynamicSmemBytes = PAIR_SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    LB_CUDA(cudaLaunchKernelEx(&cfg, pair_gemm_norm_kernel<F16>, mapA, mapB, M, N, K, tri, dNorm2, dErr));
    return LB_OK;
}

// CTA-pair (cta_group::2) launch: M % 256 == 0, N % 512 == 0; dNorm2 holds M floats.
int lb_launch_pair_gemm_norm(cudaStream_t st, const void* dA, int64_t lda, const void* dB, int64_t ldb, int64_t M, int64_t N, int64_t K,
    int tri, float* dNorm2, int* dErr, int sms, int f16)
{
    using namespace tf32q;
    if (M % (2 * BM) || N % (2 * BN) || K % 64) return LB_ERR_ARG;
    alignas(64) CUtensorMap mapA, mapB;
    int rc;
    if ((rc = make_map(&mapA, dA, M, K, lda, BM, f16 != 0))) return rc;
    if ((rc = make_map(&mapB, dB, N, K, ldb, BN / 2, f16 != 0))) return rc;
    int npairs = sms / 2;
    if (npairs > M / (2 * BM)) npairs = (int)(M / (2 * BM));
    return f16 ? launch_pair<true>(st, mapA, mapB, M, N, K, tri, dNorm2, dErr, 2 * npairs)
               : launch_pair<false>(st, mapA, mapB, M, N, K, tri, dNorm2, dErr, 2 * npairs);
}

// Split-operand launch (fp16 hi / lo planes): dA*: M x K, dB*: N x K row-major halves; M % 256 == 0, N % 256 == 0; dNorm2: M doubles.
int lb_launch_pair_split_gemm_norm(cudaStream_t st, const void* dAh, const void* dAl, int64_t lda, const void* dBh, const void* dBl, int64_t ldb,
    int64_t M, int64_t N, int64_t K, int tri, double* dNorm2, int* dErr, int sms)
{
    using namespace tf32q;
    if (M % (2 * BM) || N % BN || K % 64) return LB_ERR_ARG;
    static LbOncePerDevice attr_once;
    if (attr_once.need()) {
        LB_CUDA(cudaFuncSetAttribute(pair_split_gemm_norm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SPLIT_SMEM_BYTES));
    }
    alignas(64) CUtensorMap mAh, mAl, mBh, mBl;
    int rc;
    if ((rc = make_map(&mAh, dAh, M, K, lda, BM, true))) return rc;
    if ((rc = make_map(&mAl, dAl, M, K, lda, BM, true))) return rc;
    if ((rc = make_map(&mBh, dBh, N, K, ldb, BN / 2, true))) return rc;
    if ((rc = make_map(&mBl, dBl, N, K, ldb, BN / 2, true))) return rc;
    int npairs = sms / 2;
    if (npairs > M / (2 * BM)) npairs = (int)(M / (2 * BM));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(2 * npairs));
    cfg.blockDim = dim3(THREADS);
    cfg.dynamicSmemBytes = SPLIT_SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    LB_CUDA(cudaLaunchKernelEx(&cfg, pair_split_gemm_norm_kernel, mAh, mAl, mBh, mBl, M, N, K, tri, dNorm2, dErr));
    return LB_OK;
}

extern "C" int lb_debug_pair_gemm(const void* dA, const void* dB, long long M, long long N, long long K, int tri, float* dNorm2, int f16)
{
    int* dErr = nullptr;
    LB_CUDA(cudaMalloc(&dErr, sizeof(int)));
    LB_CUDA(cudaMemset(dErr, 0, sizeof(int)));
    int rc = lb_launch_pair_gemm_norm(0, dA, K, dB, K, M, N, K, tri, dNorm2, dErr, 148, f16);
    if (rc) { cudaFree(dErr); return rc; }
    LB_CUDA(cudaDeviceSynchronize());
    int herr = 0;
    LB_CUDA(cudaMemcpy(&herr, dErr, sizeof(int), cudaMemcpyDeviceToHost));
    cudaFree(dErr);
    return herr ? LB_ERR_TIMEOUT : LB_OK;
}

__global__ void debug_exp_kernel(const double* in, double* out, long long n)
{
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) out[i] = lb_exp_nonpos(in[i]);
}

// test hook: out[i] = lb_exp_nonpos(in[i]) (device pointers)
extern "C" int lb_debug_exp(const double* dIn, double* dOut, long long n)
{
    debug_exp_kernel<<<(unsigned)((n + 255) / 256), 256>>>(dIn, dOut, n);
    LB_CUDA(cudaGetLastError());
    LB_CUDA(cudaDeviceSynchronize());
    return LB_OK;
}

extern "C" int lb_debug_tf32_gemm_cluster(const void* dA, const void* dB, long long M, long long N, long long K, int tri, float* dNorm2,
    int cl, int f16)
{
    int* dErr = nullptr;
    LB_CUDA(cudaMalloc(&dErr, sizeof(int)));
    LB_CUDA(cudaMemset(dErr, 0, sizeof(int)));
    int rc = lb_launch_tf32_gemm_norm_cluster(0, dA, K, dB, K, M, N, K, tri, dNorm2, dErr, 148, cl, f16);
    if (rc) { cudaFree(dErr); return rc; }
    LB_CUDA(cudaDeviceSynchronize());
    int herr = 0;
    LB_CUDA(cudaMemcpy(&herr, dErr, sizeof(int), cudaMemcpyDeviceToHost));
    cudaFree(dErr);
    return herr ? LB_ERR_TIMEOUT : LB_OK;
}

extern "C" int lb_debug_tf32_gemm(const void* dA, const void* dB, long long M, long long N, long long K, int tri, float* dNorm2,
    float* dDout, int grid, int f16)
{
    int* dErr = nullptr;
    LB_CUDA(cudaMalloc(&dErr, sizeof(int)));
    LB_CUDA(cudaMemset(dErr, 0, sizeof(int)));
    int rc = lb_launch_tf32_gemm_norm(0, dA, K, dB, K, M, N, K, tri, dNorm2, dDout, dErr, grid, f16);
    if (rc) { cudaFree(dErr); return rc; }
    LB_CUDA(cudaDeviceSynchronize());
    int herr = 0;
    LB_CUDA(cudaMemcpy(&herr, dErr, sizeof(int), cudaMemcpyDeviceToHost));
    cudaFree(dErr);
    return herr ? LB_ERR_TIMEOUT : LB_OK;
}

// ===========================================================================
// TF32 prediction path: K*^T (fp32, K-major) build, mu GEMV, L^-1 cast/transposed, sigma^2 from the row norms.
// ===========================================================================
namespace tf32q {

// fp32 -> tf32 with round-to-nearest: tcgen05.mma.kind::tf32 ignores the low 13 mantissa bits of its operands, i.e. truncates;
// a truncated operand is biased low, and the bias of |L^-1 k*|^2 does not average out over the N terms of the sum.
__device__ __forceinline__ float tf32_rna(float v)
{
    uint32_t u;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(v));
    return __uint_as_float(u);
}

constexpr int DCH_WIDE = 16; // input dimensions staged per pass

// Kt[c * ldk + n] = (float) k(x_n, q_c)  for one tile of 128 candidates x 128 training points; zero for n >= N.
// grid: (Np/128, Mc/128).  Same thread mapping as kbuild_kernel: the two consecutive "rows" of a thread are two
// consecutive n, stored as one float2 (n is the contiguous, K-major index of the GEMM's A operand).
// F16: the stored values are k / sigma_f^2 (in (0, 1]) as half.  EDGE: the tile crosses N or M (zero beyond).
// Tiles [i_first, i_first + ni) x [j_first, j_first + nj) are walked with a grid-stride loop (training index fastest), so the
// same kernel runs one tile per CTA or as a small persistent grid.
// Squared distances on the fp64 TENSOR pipe: z_cn = |q_c|^2 + |x_n|^2 - 2 q_c . x_n with the cross term as an
// mma.m8n8k4.f64 (candidates = M side, training points = N side, input dimensions = K, zero padded to a multiple of 4).
// ncu on the FMA version of this kernel showed the fp64 ALU pipe 61 % active and the tensor pipe idle, and on the DMMA GEMMs
// the reverse (profiles/r01_ncu_*): the two are separate pipes, so moving the D-loop (24 of ~55 fp64 operations per pair at
// D = 12) to DMMA leaves the ALU pipe to exp / scaling / the mean and bias partials.  The cancellation costs ~1e-16 (|q|^2 +
// |x|^2) absolute on z, i.e. <= 1e-13 relative on k: inside the 1e-9 bar this path states for mu.
// A thread ends up with candidate g (+ 8 mb) x training points 2t, 2t+1 (+ 8 nb): two consecutive K-major elements = one
// half2 / float2 store.
constexpr int XP = LB_TILE + 4; // pitch of the staged point tiles: the (d = t, point = g) fragment loads of a half-warp hit 16 distinct banks

template <int KID, bool F16, bool EDGE, int DCH>
__device__ __forceinline__ void kstar_t32_body(const double* __restrict__ Xs, int64_t Np, int64_t N, const double* __restrict__ Qs, int64_t Mp,
    int64_t M, void* __restrict__ Kt_, int64_t ldk, const KernParams& kp, const double* __restrict__ alpha, int P,
    double* __restrict__ mu_part, int64_t i_first, int64_t j_first, int64_t ni, int64_t nj, const double* __restrict__ colw,
    void* __restrict__ Kt_lo = nullptr)
{
    static_assert(DCH % 4 == 0, "k4 steps");
    __shared__ __align__(128) double sxi[DCH][XP]; // training points of the tile, dimension-major
    __shared__ __align__(128) double sxj[DCH][XP]; // candidates
    __shared__ double sni[LB_TILE], snj[LB_TILE];  // squared norms of the staged coordinates
    __shared__ double spm[8][64];
    __shared__ __align__(8) uint64_t bar;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int D = kp.D;
    if (tid == 0) {
        lb_mbar_init(&bar, 1);
        lb_fence_barrier_init();
    }
    __syncthreads();
    uint32_t phase = 0;
    const int npass = (D + DCH - 1) / DCH;
    for (int64_t tile = blockIdx.x; tile < ni * nj; tile += gridDim.x) {
    const int64_t ti = i_first + tile % ni; // training tile index (also the slot of the mean partial)
    const int64_t i0 = ti * LB_TILE, j0 = (j_first + tile / ni) * LB_TILE; // i: training, j: candidates
    __syncthreads(); // the previous tile's epilogue has read the norms
    if (tid < LB_TILE) sni[tid] = 0.0;
    else snj[tid - LB_TILE] = 0.0;
    for (int h = 0; h < 2; ++h) {
        double acc[8][2][2]; // [candidate block mb][training block nb][2 consecutive training points]
#pragma unroll
        for (int mb = 0; mb < 8; ++mb)
#pragma unroll
            for (int nb = 0; nb < 2; ++nb) acc[mb][nb][0] = acc[mb][nb][1] = 0.0;
        for (int pass = 0; pass < npass; ++pass) {
            const int d0 = pass * DCH;
            const int dc = min(DCH, D - d0), dc4 = (dc + 3) & ~3;
            if (!(npass == 1 && h == 1)) {
                __syncthreads();
                if (tid == 0) {
                    lb_fence_proxy_async();
                    lb_mbar_expect_tx(&bar, (uint32_t)(2 * dc * LB_TILE * sizeof(double)));
                    for (int d = 0; d < dc; ++d) {
                        lb_bulk_g2s(&sxi[d][0], Xs + (int64_t)(d0 + d) * Np + i0, LB_TILE * sizeof(double), &bar);
                        lb_bulk_g2s(&sxj[d][0], Qs + (int64_t)(d0 + d) * Mp + j0, LB_TILE * sizeof(double), &bar);
                    }
                }
                for (int d = dc; d < dc4; ++d) { // zero rows up to the k4 boundary
                    if (tid < LB_TILE) sxi[d][tid] = 0.0;
                    else sxj[d][tid - LB_TILE] = 0.0;
                }
                lb_mbar_wait(&bar, phase);
                phase ^= 1;
                if (h == 0) { // squared norms, accumulated over the passes (one point per thread)
                    double s = 0.0;
                    if (tid < LB_TILE) {
                        for (int d = 0; d < dc; ++d) s = fma(sxi[d][tid], sxi[d][tid], s);
                        sni[tid] += s;
                    }
                    else {
                        for (int d = 0; d < dc; ++d) s = fma(sxj[d][tid - LB_TILE], sxj[d][tid - LB_TILE], s);
                        snj[tid - LB_TILE] += s;
                    }
                }
                __syncthreads();
            }
            for (int ks = 0; ks < dc4; ks += 4) {
                const double b0 = sxi[ks + t][warp * 16 + g], b1 = sxi[ks + t][warp * 16 + 8 + g];
#pragma unroll
                for (int mb = 0; mb < 8; ++mb) {
                    const double a = sxj[ks + t][h * 64 + mb * 8 + g];
                    lb_dmma_8x8x4(acc[mb][0][0], acc[mb][0][1], a, b0);
                    lb_dmma_8x8x4(acc[mb][1][0], acc[mb][1][1], a, b1);
                }
            }
        }
        // kernel values (kept in acc for the partial sums), K-major stores
#pragma unroll
        for (int mb = 0; mb < 8; ++mb) {
            const int cl = h * 64 + mb * 8 + g; // candidate within the tile
            const int64_t gj = j0 + cl;
            const double nq = snj[cl];
#pragma unroll
            for (int nb = 0; nb < 2; ++nb) {
                const int tl = warp * 16 + nb * 8 + 2 * t; // training point within the tile (even)
                const int64_t gi = i0 + tl;
                float v[2];
                double uu[2];
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const double z = fmax(nq + sni[tl + e] - 2.0 * acc[mb][nb][e], 0.0);
                    double u = lb_unit_kernel_from_z<KID>(z, kp);
                    if (EDGE) {
                        if (gi + e >= N || gj >= M) u = 0.0;
                    }
                    const double k = kp.sf2 * u;
                    acc[mb][nb][e] = k;
                    uu[e] = u;
                    v[e] = (float)(F16 ? u : k);
                }
                if (F16) {
                    const __half2 hi = __floats2half2_rn(v[0], v[1]);
                    *reinterpret_cast<__half2*>(reinterpret_cast<__half*>(Kt_) + gj * ldk + gi) = hi;
                    if (Kt_lo) { // split operands (LB_PREC_FP16X3): lo = (u - hi) * 2^11, the next 11 bits of the value
                        const float2 hf = __half22float2(hi);
                        *reinterpret_cast<__half2*>(reinterpret_cast<__half*>(Kt_lo) + gj * ldk + gi)
                            = __floats2half2_rn((float)((uu[0] - (double)hf.x) * 2048.0), (float)((uu[1] - (double)hf.y) * 2048.0));
                    }
                }
                else *reinterpret_cast<float2*>(reinterpret_cast<float*>(Kt_) + gj * ldk + gi) = make_float2(tf32_rna(v[0]), tf32_rna(v[1]));
            }
        }
        // mean partials from the fp64 kernel values: mu_part[(p * ntiles + tile) * Mp + candidate] = sum over this tile's
        // 128 training points (lanes -> warps in a fixed order; the tiles are summed in order by mu_reduce_kernel).
        // Pass p == P (when colw != nullptr): sum_k k*_k^2 |L^-1 e_k|^2, the weight of the rounding-noise bias of |L^-1 k*|^2
        // (sigma2_t32_kernel subtracts its expectation).
        for (int p = 0; p < P + (colw ? 1 : 0); ++p) {
            const bool bias = (p == P);
            const double* wv = (bias ? colw : alpha + (int64_t)p * Np) + i0 + warp * 16 + 2 * t;
            const double w00 = wv[0], w01 = wv[1], w10 = wv[8], w11 = wv[9];
#pragma unroll
            for (int mb = 0; mb < 8; ++mb) {
                double sm;
                if (bias)
                    sm = fma(acc[mb][0][0] * acc[mb][0][0], w00, fma(acc[mb][0][1] * acc[mb][0][1], w01,
                        fma(acc[mb][1][0] * acc[mb][1][0], w10, acc[mb][1][1] * acc[mb][1][1] * w11)));
                else
                    sm = fma(acc[mb][0][0], w00, fma(acc[mb][0][1], w01, fma(acc[mb][1][0], w10, acc[mb][1][1] * w11)));
                sm += __shfl_xor_sync(0xffffffffu, sm, 1);
                sm += __shfl_xor_sync(0xffffffffu, sm, 2);
                if (t == 0) spm[warp][mb * 8 + g] = sm;
            }
            __syncthreads();
            if (tid < 64) {
                double sacc = spm[0][tid];
#pragma unroll
                for (int w = 1; w < 8; ++w) sacc += spm[w][tid];
                mu_part[((int64_t)p * (Np / LB_TILE) + ti) * Mp + j0 + h * 64 + tid] = sacc;
            }
            __syncthreads();
        }
    }
    } // tile loop
}

// one tile per CTA (or any grid): two CTAs per SM by registers
template <int KID, bool F16, bool EDGE, int DCH>
__global__ void __launch_bounds__(256, 2)
kstar_t32_kernel(const double* __restrict__ Xs, int64_t Np, int64_t N, const double* __restrict__ Qs, int64_t Mp, int64_t M,
    void* __restrict__ Kt_, int64_t ldk, KernParams kp, const double* __restrict__ alpha, int P,
    double* __restrict__ mu_part, int64_t i_first, int64_t j_first, int64_t ni, int64_t nj, const double* __restrict__ colw,
    void* __restrict__ Kt_lo)
{
    kstar_t32_body<KID, F16, EDGE, DCH>(Xs, Np, N, Qs, Mp, M, Kt_, ldk, kp, alpha, P, mu_part, i_first, j_first, ni, nj, colw, Kt_lo);
}
// mu[c*P + p] = sum over the training tiles of the partials written by kstar_t32_kernel (fixed order)
__global__ void __launch_bounds__(256)
mu_reduce_kernel(const double* __restrict__ part, int ntiles, int64_t Mp, int P, int64_t M, double* __restrict__ mu,
    double* __restrict__ bias)
{
    const int64_t c = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (c >= M) return;
    for (int p = 0; p < P + (bias ? 1 : 0); ++p) {
        const double* q = part + (int64_t)p * ntiles * Mp + c;
        double s = 0.0;
        for (int t = 0; t < ntiles; ++t) s += q[(int64_t)t * Mp];
        if (p < P) mu[c * P + p] = s;
        else bias[c] = s;
    }
}

// w[k] = sum_n Linv[n, k]^2 (column k of the lower-triangular inverse, column-major): one block per column
__global__ void __launch_bounds__(256)
colnorm2_kernel(const double* __restrict__ Linv, int64_t ld, double* __restrict__ w)
{
    __shared__ double red[8];
    const int64_t k = blockIdx.x;
    const double* col = Linv + k * ld;
    double s = 0.0;
    for (int64_t n = k + threadIdx.x; n < ld; n += 256) s = fma(col[n], col[n], s);
    s = lb_warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < 8; ++i) t += red[i];
        w[k] = t;
    }
}

// max |Linv| (for the fp16 scale): one value per block, reduced on the host (tiny)
__global__ void __launch_bounds__(256)
absmax_kernel(const double* __restrict__ A, int64_t n, double* __restrict__ out)
{
    __shared__ double red[8];
    double m = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) m = fmax(m, fabs(A[i]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) m = fmax(m, red[w]);
        out[blockIdx.x] = m;
    }
}

// LinvR[n * ldr + k] = (float) Linv[n + k * ld]  (column-major fp64 -> row-major fp32, 32 x 32 smem transpose)
template <bool F16>
__global__ void __launch_bounds__(256)
linv_to_rowmajor_kernel(const double* __restrict__ Linv, int64_t ld, void* __restrict__ R_, int64_t ldr, double scale, void* __restrict__ Rlo_)
{
    __shared__ double tile[32][33];
    const int64_t n0 = (int64_t)blockIdx.x * 32, k0 = (int64_t)blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int kk = ty; kk < 32; kk += 8) tile[kk][tx] = (k0 + kk <= n0 + tx) ? Linv[n0 + tx + (k0 + kk) * ld] * scale : 0.0;
    __syncthreads();
    for (int nn = ty; nn < 32; nn += 8) {
        const double v = tile[tx][nn];
        if (F16) {
            const __half hi = __float2half_rn((float)v);
            reinterpret_cast<__half*>(R_)[(n0 + nn) * ldr + k0 + tx] = hi;
            if (Rlo_) reinterpret_cast<__half*>(Rlo_)[(n0 + nn) * ldr + k0 + tx] = __float2half_rn((float)((v - (double)__half2float(hi)) * 2048.0));
        }
        else reinterpret_cast<float*>(R_)[(n0 + nn) * ldr + k0 + tx] = tf32_rna((float)v);
    }
}

// ---- inversion spread over G GPUs (query.cu: lb_launch_linv_columns): pack this rank's columns, adopt everybody's ----------------
// V: Np x ldr column-major, local column tile t = global tile c = rank + t * G.  Chunk of a rank (what the all_gather moves):
//   [ hi plane: Np x ldr row-major (fp16, or fp32 holding tf32) | lo plane (split mode only) | w: ldr doubles = |L^-1 e_k|^2 ]
template <bool F16>
__global__ void __launch_bounds__(256)
linv_cols_pack_kernel(const double* __restrict__ V, int64_t ld, int rank, int G, int T, void* __restrict__ R_, int64_t ldr, double scale,
    void* __restrict__ Rlo_)
{
    __shared__ double tile[32][33];
    const int64_t n0 = (int64_t)blockIdx.x * 32, l0 = (int64_t)blockIdx.y * 32; // rows, local columns
    const int64_t c = rank + (l0 / LB_TILE) * G;                                  // global column tile
    const int64_t k0 = c * LB_TILE + (l0 % LB_TILE);                              // global column of local column l0
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int kk = ty; kk < 32; kk += 8) tile[kk][tx] = (c < T && k0 + kk <= n0 + tx) ? V[n0 + tx + (l0 + kk) * ld] * scale : 0.0;
    __syncthreads();
    for (int nn = ty; nn < 32; nn += 8) {
        const double v = tile[tx][nn];
        if (F16) {
            const __half hi = __float2half_rn((float)v);
            reinterpret_cast<__half*>(R_)[(n0 + nn) * ldr + l0 + tx] = hi;
            if (Rlo_) reinterpret_cast<__half*>(Rlo_)[(n0 + nn) * ldr + l0 + tx] = __float2half_rn((float)((v - (double)__half2float(hi)) * 2048.0));
        }
        else reinterpret_cast<float*>(R_)[(n0 + nn) * ldr + l0 + tx] = tf32_rna((float)v);
    }
}

// w[l] = sum_n V[n, l]^2 (rows above the diagonal are zeros): one block per local column
__global__ void __launch_bounds__(256)
colnorm2_cols_kernel(const double* __restrict__ V, int64_t ld, double* __restrict__ w)
{
    __shared__ double red[8];
    const double* col = V + (int64_t)blockIdx.x * ld;
    double s = 0.0;
    for (int64_t n = threadIdx.x; n < ld; n += 256) s = fma(col[n], col[n], s);
    s = lb_warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < 8; ++i) t += red[i];
        w[blockIdx.x] = t;
    }
}

// out[n, c * 128 + kk] = plane of rank (c mod G), row n, local column (c / G) * 128 + kk; 16-byte pieces, one block per row
__global__ void __launch_bounds__(256)
linv_unpermute_kernel(const char* __restrict__ all, size_t chunk_bytes, size_t plane_off, int G, int T, int64_t Np, int64_t ldr, int esz,
    char* __restrict__ out)
{
    const int64_t n = blockIdx.x;
    const int tile_bytes = LB_TILE * esz, per_tile = tile_bytes / 16;
    for (int idx = threadIdx.x; idx < T * per_tile; idx += 256) {
        const int c = idx / per_tile, q = idx - c * per_tile;
        const char* src = all + (size_t)(c % G) * chunk_bytes + plane_off + ((size_t)n * ldr + (size_t)(c / G) * LB_TILE) * esz + (size_t)q * 16;
        char* dst = out + ((size_t)n * Np + (size_t)c * LB_TILE) * esz + (size_t)q * 16;
        *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(src);
    }
}

__global__ void __launch_bounds__(256)
linvw_unpermute_kernel(const char* __restrict__ all, size_t chunk_bytes, size_t w_off, int G, int64_t Np, double* __restrict__ w)
{
    const int64_t k = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (k >= Np) return;
    const int64_t c = k / LB_TILE, kk = k % LB_TILE;
    w[k] = reinterpret_cast<const double*>(all + (size_t)(c % G) * chunk_bytes + w_off)[(c / G) * LB_TILE + kk];
}

// sigma^2 from fp64 norms (split-operand mode): no rounding-bias term
__global__ void __launch_bounds__(256)
sigma2_split_kernel(const double* __restrict__ norm2, int64_t M, double kvv, double noise, double norm_unscale, double* __restrict__ s2)
{
    const int64_t c = blockIdx.x * (int64_t)256 + threadIdx.x;
    if (c >= M) return;
    double res = kvv - norm2[c] * norm_unscale;
    res = (res <= 2.220446049250313e-16) ? 0.0 : res; // gp.hpp:623
    s2[c] = res + noise;                               // gp.hpp:166
}

__global__ void __launch_bounds__(256)
sigma2_t32_kernel(const float* __restrict__ norm2, int nparts, int64_t part_stride, int64_t M, double kvv, double noise,
    double norm_unscale, const double* __restrict__ bias, double bias_coeff, double* __restrict__ s2)
{
    const int64_t c = blockIdx.x * (int64_t)256 + threadIdx.x;
    if (c >= M) return;
    double nrm = 0.0;
    for (int p = 0; p < nparts; ++p) nrm += (double)norm2[(int64_t)p * part_stride + c]; // partial sums of the cluster's CTAs
    // Rounding both operands to an 11-bit significand adds zero-mean noise e_n to every D[c, n]; sum_n D^2 then carries the
    // positive bias E sum e_n^2 = 2 u_r^2 sum_k k*_k^2 |L^-1 e_k|^2 (u_r^2 = E[relative rounding error^2]), which grows with
    // cond(K) while the zero-mean part does not (DESIGN.md §4.5): subtract its expectation.
    double res = kvv - (nrm * norm_unscale - (bias ? bias_coeff * bias[c] : 0.0));
    res = (res <= 2.220446049250313e-16) ? 0.0 : res; // gp.hpp:623
    s2[c] = res + noise;                               // gp.hpp:166
}

} // namespace tf32q

int lb_launch_linv(lb_gp* h);


// CTAs per cluster sharing one candidate tile (A operand multicast).  Measured at N=16384, 1M candidates: 1 -> 518 ms,
// 2 -> 467 ms, 4 -> 726 ms (lock-step coupling of four CTAs costs more than the saved HBM stream): default 2;
// LB_TF32_CLUSTER=1|2|4 overrides.
int lb_tf32_cluster_size()
{
    static int cl = 0;
    if (!cl) {
        const char* e = getenv("LB_TF32_CLUSTER");
        cl = e ? atoi(e) : 2;
        if (cl != 1 && cl != 2 && cl != 4) cl = 2;
    }
    return cl;
}

// CTA-pair kernel (cta_group::2, pair_gemm_norm_kernel) unless LB_TF32_PAIR=0: config 4 fp16 GEMM 229 -> see DESIGN.md §4.5
int lb_tf32_pair_mode()
{
    static int pm = -1;
    if (pm < 0) {
        const char* e = getenv("LB_TF32_PAIR");
        pm = e ? (atoi(e) != 0) : 1;
    }
    return pm;
}

// Prepare the row-major reduced-precision copy of L^-1 (rows padded with zeros to a multiple of 256 * cluster size).
// fp32 (tf32 MMA) stores L^-1 as is; fp16 stores L^-1 * 2^e with e chosen so that max |.| <= 2^14.
int lb_tf32_prepare(lb_gp* h)
{
    using namespace tf32q;
    if (h->linv32_valid) return LB_OK;
    const bool split = (h->precision == 3); // fp16 hi / lo planes (LB_PREC_FP16X3)
    const bool f16 = (h->precision == 2) || split;
    int rc;
    if (!h->linv_valid && (rc = lb_launch_linv(h))) return rc;
    const int cl = lb_tf32_pair_mode() ? 2 : lb_tf32_cluster_size(); // the pair kernel walks two 256-row n-tiles per group
    const int64_t Np = h->Np, Nr = (Np + BN * cl - 1) / (BN * cl) * (BN * cl);
    const size_t esz = split ? 4 : (f16 ? 2 : 4); // split: two fp16 planes of Nr x Np
    if (!h->dLinv32 || h->linv32_rows != Nr) {
        lb_dfree_sync(h, h->dLinv32);
        h->dLinv32 = nullptr;
        LB_ALLOC(h, h->dLinv32, esz * Nr * Np);
        h->linv32_rows = Nr;
    }
    double scale = 1.0;
    if (f16) {
        if ((rc = lb_ensure_scratch(h, sizeof(double) * 1024))) return rc;
        absmax_kernel<<<1024, 256, 0, h->stream>>>(h->dLinv, Np * Np, h->dScratch);
        h->launches++;
        double part[1024];
        LB_CUDA(cudaMemcpyAsync(part, h->dScratch, sizeof(part), cudaMemcpyDeviceToHost, h->stream));
        LB_CUDA(cudaStreamSynchronize(h->stream));
        double mx = 0.0;
        for (double v : part) mx = v > mx ? v : mx;
        if (!(mx > 0.0) || !std::isfinite(mx)) return LB_ERR_STATE;
        scale = std::ldexp(1.0, 14 - (int)std::ceil(std::log2(mx)));
    }
    h->linv32_scale = scale;
    __half* lo_plane = split ? reinterpret_cast<__half*>(h->dLinv32) + Nr * Np : nullptr;
    if (split) LB_CUDA(cudaMemsetAsync(h->dLinv32, 0, esz * Nr * Np, h->stream)); // both planes incl. the padding rows
    else if (Nr > Np) LB_CUDA(cudaMemsetAsync((char*)h->dLinv32 + esz * Np * Np, 0, esz * (Nr - Np) * Np, h->stream));
    dim3 grid((unsigned)(Np / 32), (unsigned)(Np / 32));
    LbProfScope ps(h, h->stream, LB_PC_OTHER);
    if (f16) linv_to_rowmajor_kernel<true><<<grid, 256, 0, h->stream>>>(h->dLinv, Np, h->dLinv32, Np, scale, lo_plane);
    else linv_to_rowmajor_kernel<false><<<grid, 256, 0, h->stream>>>(h->dLinv, Np, h->dLinv32, Np, 1.0, nullptr);
    h->launches++;
    if (!h->dLinvW || h->linvw_np != Np) {
        lb_dfree_sync(h, h->dLinvW);
        h->dLinvW = nullptr;
        LB_ALLOC(h, h->dLinvW, sizeof(double) * Np);
        h->linvw_np = Np;
    }
    colnorm2_kernel<<<(unsigned)Np, 256, 0, h->stream>>>(h->dLinv, Np, h->dLinvW); // weights of the rounding-bias correction
    h->launches++;
    LB_CUDA(cudaGetLastError());
    h->linv32_valid = true;
    return LB_OK;
}

// ---- the same copy assembled from the column chunks of G ranks (lb_dinv_* in abi.cu; limbo_b200/dist_inv.py) --------------------
int64_t lb_linv_columns_width(const lb_gp* h, int G);

static size_t dinv_plane_bytes(const lb_gp* h, int G)
{
    const bool f16 = (h->precision == 2) || (h->precision == 3);
    return (size_t)h->Np * (size_t)lb_linv_columns_width(h, G) * (f16 ? 2 : 4);
}

size_t lb_dinv_chunk_bytes_impl(const lb_gp* h, int G)
{
    return dinv_plane_bytes(h, G) * (h->precision == 3 ? 2 : 1) + sizeof(double) * (size_t)lb_linv_columns_width(h, G);
}

// max |V| over this rank's columns (host value; synchronises the handle's stream)
int lb_dinv_absmax(lb_gp* h, const double* dV, int G, double* out)
{
    using namespace tf32q;
    int rc;
    if ((rc = lb_ensure_scratch(h, sizeof(double) * 1024))) return rc;
    absmax_kernel<<<1024, 256, 0, h->stream>>>(dV, h->Np * lb_linv_columns_width(h, G), h->dScratch);
    h->launches++;
    double part[1024];
    LB_CUDA(cudaMemcpyAsync(part, h->dScratch, sizeof(part), cudaMemcpyDeviceToHost, h->stream));
    LB_CUDA(cudaStreamSynchronize(h->stream));
    double mx = 0.0;
    for (double v : part) mx = v > mx ? v : mx;
    *out = mx;
    return LB_OK;
}

// the fp16 scale lb_tf32_prepare derives from max |L^-1| (1 for tf32)
static int dinv_scale(const lb_gp* h, double absmax, double* scale)
{
    *scale = 1.0;
    if (h->precision == 2 || h->precision == 3) {
        if (!(absmax > 0.0) || !std::isfinite(absmax)) return LB_ERR_STATE;
        *scale = std::ldexp(1.0, 14 - (int)std::ceil(std::log2(absmax)));
    }
    return LB_OK;
}

int lb_dinv_pack_impl(lb_gp* h, const double* dV, int rank, int G, double absmax_all, void* dChunk)
{
    using namespace tf32q;
    const bool split = (h->precision == 3), f16 = (h->precision == 2) || split;
    const int64_t Np = h->Np, ldr = lb_linv_columns_width(h, G);
    const int T = (int)(Np / LB_TILE);
    double scale;
    int rc = dinv_scale(h, absmax_all, &scale);
    if (rc) return rc;
    char* base = reinterpret_cast<char*>(dChunk);
    const size_t plane = dinv_plane_bytes(h, G);
    dim3 grid((unsigned)(Np / 32), (unsigned)(ldr / 32));
    LbProfScope ps(h, h->stream, LB_PC_OTHER);
    if (f16) linv_cols_pack_kernel<true><<<grid, 256, 0, h->stream>>>(dV, Np, rank, G, T, base, ldr, scale, split ? base + plane : nullptr);
    else linv_cols_pack_kernel<false><<<grid, 256, 0, h->stream>>>(dV, Np, rank, G, T, base, ldr, 1.0, nullptr);
    colnorm2_cols_kernel<<<(unsigned)ldr, 256, 0, h->stream>>>(dV, Np, reinterpret_cast<double*>(base + plane * (split ? 2 : 1)));
    h->launches += 2;
    LB_CUDA(cudaGetLastError());
    return LB_OK;
}

int lb_dinv_adopt_impl(lb_gp* h, int G, const void* dAll, double absmax_all)
{
    using namespace tf32q;
    const bool split = (h->precision == 3), f16 = (h->precision == 2) || split;
    const int cl = lb_tf32_pair_mode() ? 2 : lb_tf32_cluster_size();
    const int64_t Np = h->Np, Nr = (Np + BN * cl - 1) / (BN * cl) * (BN * cl), ldr = lb_linv_columns_width(h, G);
    const int T = (int)(Np / LB_TILE);
    const size_t esz = split ? 4 : (f16 ? 2 : 4), el = f16 ? 2 : 4;
    double scale;
    int rc = dinv_scale(h, absmax_all, &scale);
    if (rc) return rc;
    if (!h->dLinv32 || h->linv32_rows != Nr) {
        lb_dfree_sync(h, h->dLinv32);
        h->dLinv32 = nullptr;
        LB_ALLOC(h, h->dLinv32, esz * Nr * Np);
        h->linv32_rows = Nr;
    }
    if (!h->dLinvW || h->linvw_np != Np) {
        lb_dfree_sync(h, h->dLinvW);
        h->dLinvW = nullptr;
        LB_ALLOC(h, h->dLinvW, sizeof(double) * Np);
        h->linvw_np = Np;
    }
    h->linv32_scale = scale;
    const size_t chunk = lb_dinv_chunk_bytes_impl(h, G), plane = dinv_plane_bytes(h, G);
    const char* all = reinterpret_cast<const char*>(dAll);
    char* out = reinterpret_cast<char*>(h->dLinv32);
    LbProfScope ps(h, h->stream, LB_PC_OTHER);
    if (Nr > Np) { // padding rows of both planes
        LB_CUDA(cudaMemsetAsync(out + el * Np * Np, 0, el * (Nr - Np) * Np, h->stream));
        if (split) LB_CUDA(cudaMemsetAsync(out + el * Nr * Np + el * Np * Np, 0, el * (Nr - Np) * Np, h->stream));
    }
    linv_unpermute_kernel<<<(unsigned)Np, 256, 0, h->stream>>>(all, chunk, 0, G, T, Np, ldr, (int)el, out);
    if (split) linv_unpermute_kernel<<<(unsigned)Np, 256, 0, h->stream>>>(all, chunk, plane, G, T, Np, ldr, (int)el, out + el * Nr * Np);
    linvw_unpermute_kernel<<<(unsigned)((Np + 255) / 256), 256, 0, h->stream>>>(all, chunk, plane * (split ? 2 : 1), G, Np, h->dLinvW);
    h->launches += split ? 3 : 2;
    LB_CUDA(cudaGetLastError());
    h->linv32_valid = true;
    return LB_OK;
}

// K*^T chunk (reduced precision, K-major) and mu (M x P, fp64) for Mc candidates.
// (Tried and dropped: running this build for chunk i+1 on a second stream under the tcgen05 GEMM of chunk i.  Even with a
// 13 KB / 104-register variant, cp.async staging, dynamic tile hand-out, polite mbarrier waits and the full 228 KB carve-out on
// the GEMM, the fp64 CTAs made almost no progress while the GEMM CTA was resident and slowed it by 15 %: 272-285 ms per 1M
// candidates against 256 ms for plain back-to-back launches, profiles/r01_config4_notes.txt.)
int lb_launch_kstar_tf32(const lb_gp* h, cudaStream_t st, int64_t Mc, const double* dQs, int64_t Mcp, float* dKt, double* dMuPart,
    double* dMu, double* dBias, long long* launches)
{
    using namespace tf32q;
    const bool split = (h->precision == 3);
    const bool f16 = (h->precision == 2) || split;
    const int64_t Np = h->Np;
    void* dKtLo = split ? (void*)(reinterpret_cast<__half*>(dKt) + Mcp * Np) : nullptr; // lo plane behind the hi plane of this chunk
    {
        LbProfScope ps(h, st, LB_PC_KSTAR);
        // interior tiles without bounds checks; the last tile row / column (when N or Mc is not a multiple of 128) with
        const int64_t nti = Np / LB_TILE, ntj = Mcp / LB_TILE;
        const int64_t fi = h->N / LB_TILE, fj = Mc / LB_TILE; // number of full tiles
        auto go = [&](auto kid, auto f16c, auto edgec, int64_t ia, int64_t ib, int64_t ja, int64_t jb) {
            if (ib <= ia || jb <= ja) return;
            const int64_t tiles = (ib - ia) * (jb - ja);
            kstar_t32_kernel<decltype(kid)::value, decltype(f16c)::value, decltype(edgec)::value, DCH_WIDE><<<(unsigned)tiles, 256, 0, st>>>(h->dXs, Np,
                h->N, dQs, Mcp, Mc, dKt, Np, h->kp, h->dAlpha, h->P, dMuPart, ia, ja, ib - ia, jb - ja, dBias ? h->dLinvW : nullptr, dKtLo);
            if (launches) ++*launches;
        };
        auto go_prec = [&](auto kid) {
            auto run = [&](auto f16c) {
                go(kid, f16c, std::false_type{}, 0, fi, 0, fj);
                go(kid, f16c, std::true_type{}, fi, nti, 0, ntj);
                go(kid, f16c, std::true_type{}, 0, fi, fj, ntj);
            };
            if (f16) run(std::true_type{});
            else run(std::false_type{});
        };
        switch (h->kp.id) {
        case LB_K_SE_ARD: go_prec(std::integral_constant<int, LB_K_SE_ARD>{}); break;
        case LB_K_MATERN52: go_prec(std::integral_constant<int, LB_K_MATERN52>{}); break;
        case LB_K_MATERN32: go_prec(std::integral_constant<int, LB_K_MATERN32>{}); break;
        default: go_prec(std::integral_constant<int, LB_K_EXP>{}); break;
        }
    }
    {
        LbProfScope ps(h, st, LB_PC_QREDUCE);
        mu_reduce_kernel<<<(unsigned)((Mc + 255) / 256), 256, 0, st>>>(dMuPart, (int)(Np / LB_TILE), Mcp, h->P, Mc, dMu, dBias);
    }
    if (launches) ++*launches;
    LB_CUDA(cudaGetLastError());
    return LB_OK;
}

// sigma2 (M, fp64 container of a reduced-precision value) from a K*^T chunk: tcgen05 GEMM + row norms, then the clamp / noise of gp.hpp:618-624
int lb_launch_sigma_tf32(const lb_gp* h, cudaStream_t st, int64_t Mc, int64_t Mcp, const float* dKt, float* dNorm2, int* dErr,
    const double* dBias, double* dS2, long long* launches)
{
    using namespace tf32q;
    const bool split = (h->precision == 3);
    const bool f16 = (h->precision == 2) || split;
    const int64_t Np = h->Np;
    const double kscale = f16 ? 1.0 / h->kp.sf2 : 1.0;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
    int rc;
    if (split) { // hi / lo planes, three MMAs per k-step, fp64 combination and norm (dNorm2 holds Mcp doubles)
        if (Mcp % (2 * BM) || h->linv32_rows % BN) return LB_ERR_ARG;
        const __half* Ah = reinterpret_cast<const __half*>(dKt);
        const __half* Bh = reinterpret_cast<const __half*>(h->dLinv32);
        {
            LbProfScope ps(h, st, LB_PC_QSTEP);
            rc = lb_launch_pair_split_gemm_norm(st, Ah, Ah + Mcp * Np, Np, Bh, Bh + h->linv32_rows * Np, Np, Mcp, h->linv32_rows, Np, 1,
                reinterpret_cast<double*>(dNorm2), dErr, sms);
        }
        if (rc) return rc;
        const double un = 1.0 / ((kscale * h->linv32_scale) * (kscale * h->linv32_scale));
        sigma2_split_kernel<<<(unsigned)((Mc + 255) / 256), 256, 0, st>>>(reinterpret_cast<const double*>(dNorm2), Mc, h->kp.sf2, h->kp.noise, un, dS2);
        if (launches) *launches += 2;
        LB_CUDA(cudaGetLastError());
        return LB_OK;
    }
    const bool pair = lb_tf32_pair_mode() && (Mcp % (2 * BM) == 0) && (h->linv32_rows % (2 * BN) == 0);
    const int cl = pair ? 1 : lb_tf32_cluster_size(); // number of partial norms per candidate
    {
        LbProfScope ps(h, st, LB_PC_QSTEP);
        if (pair) rc = lb_launch_pair_gemm_norm(st, dKt, Np, h->dLinv32, Np, Mcp, h->linv32_rows, Np, 1, dNorm2, dErr, sms, f16);
        else if (cl == 1) rc = lb_launch_tf32_gemm_norm(st, dKt, Np, h->dLinv32, Np, Mcp, h->linv32_rows, Np, 1, dNorm2, nullptr, dErr, sms, f16);
        else rc = lb_launch_tf32_gemm_norm_cluster(st, dKt, Np, h->dLinv32, Np, Mcp, h->linv32_rows, Np, 1, dNorm2, dErr, sms, cl, f16);
    }
    if (rc) return rc;
    // D was computed from (K* kscale) and (L^-1 scale): |V|^2 = norm / (kscale scale)^2
    const double unscale = 1.0 / ((kscale * h->linv32_scale) * (kscale * h->linv32_scale));
    // u_r^2 for round-to-nearest with an 11-bit significand and log-uniform mantissas: (2^-22 / 3) * 0.541; both operands: x 2
    const double bias_coeff = 2.0 * (1.0 / 4194304.0 / 3.0) * 0.541;
    sigma2_t32_kernel<<<(unsigned)((Mc + 255) / 256), 256, 0, st>>>(dNorm2, cl, Mcp, Mc, h->kp.sf2, h->kp.noise, unscale, dBias, bias_coeff, dS2);
    if (launches) *launches += 2;
    LB_CUDA(cudaGetLastError());
    return LB_OK;
}
