// limbo_b200/csrc/query_i8.cu — the trailing update of the panel query (query.cu, namespace panel) as exact int8 digit
// products on the 5th-generation tensor cores (Ozaki scheme).
//
//     T_s = K*_s - L[s, 0:s] V[0:s]          (super-block s of 2048 rows, K = s * 2048)
//
// fp64 has no tcgen05 kind and DMMA shares its datapath with DFMA, so on the fp64 pipe this GEMM cannot get faster than the
// DMMA roof.  Here both operands are split into S = 7 signed base-2^7 digit planes,
//     L[r, k] = 2^(e_r - 6) sum_i a_i[r, k] 2^(-7 i)        e_r: per row, |L[r, :]| < 2^e_r
//     V[k, c] = 2^(e_V - 6) sum_j b_j[k, c] 2^(-7 j)        e_V: fixed, |V| <= |V_c| <= sigma_f < 2^e_V  (k*^T K^-1 k* <= k(v,v))
// with round-to-nearest digits (|a|, |b| <= 64), and only the 28 pairs with i + j < S are formed.  Pairs of the same digit sum
// g = i + j go to one int32 TMEM accumulator: |acc_g| <= S * 64^2 * K < 2^31 for K <= MAX_K = 74898, so the products are exact and
//     L V = 2^(e_r + e_V) sum_g 2^(-12 - 7 g) acc_g
// is recombined in fp64 (smallest group first).  The truncation (pairs with i + j >= S and the last digits) costs ~1e-13 on
// sigma^2 at N = 16384 (tests/test_query_int8_numerics.py restates the arithmetic in numpy).
//
// Digit planes of L (the strictly block-lower rectangles L[s, 0:s] of the super-blocks, row-major, one int32 exponent per row) are
// built once per factorisation (lb_ldig_prepare); the digit planes of V are cut from each solved super-block (vdig_split_kernel).
#include "tcgen05.cuh"
#include <climits>
#include <cmath>
#include <cstdlib>

namespace qi8 {

using namespace lbtc;

constexpr int S = 7;                  // digit slices per operand
constexpr int SB_ROWS = 2048;         // rows of a super-block of the panel query (panel::SB * LB_TILE)
constexpr int BM = 128;               // rows of L per tile (UMMA M, TMEM lanes)
constexpr int BN = 64;                // candidates per tile (UMMA N): S accumulators of BN columns = 448 of the 512 TMEM columns
constexpr int BK = 64;                // k per stage: 64-byte rows, SWIZZLE_64B; two MMAs (K = 32) per digit pair
constexpr int STAGES = 2;
constexpr int A_PLANE = BM * BK;      // 8 KB
constexpr int B_PLANE = BN * BK;      // 4 KB
constexpr int A_BYTES = S * A_PLANE;  // 56 KB
constexpr int STAGE_BYTES = S * (A_PLANE + B_PLANE); // 84 KB
constexpr int THREADS = 192;
constexpr size_t SMEM_BYTES = (size_t)STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;
constexpr int64_t MAX_K = 74898;      // S * 64^2 * K < 2^31

// K-major, SWIZZLE_64B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address >> 4 | LBO (unused) = 1 |
// SBO = 8 rows x 64 B = 512 B -> 32 | version 1 | layout 4 (SWIZZLE_64B)
__device__ __forceinline__ uint64_t desc_sw64(uint32_t smem_addr)
{
    return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | (1ull << 16) | (32ull << 32) | (1ull << 46) | (4ull << 61);
}
// instruction descriptor, kind::i8: D = S32 (2 @4), A / B signed int8 (1 @7 / @10), both K-major, N >> 3 @17, M >> 4 @24
constexpr uint32_t IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

__device__ __forceinline__ void umma_i8(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(IDESC), "r"(accumulate)
        : "memory");
}
// all S planes of one operand tile in one copy: box {BK bytes, rows, S planes}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
                     lb_smem_u32(dst)),
                 "l"(map), "r"(c0), "r"(c1), "r"(0), "r"(lb_smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}

// S signed digits of x (|x| < 64 after scaling), packed little-endian: byte j of word w = digit of element 4 w + j
__device__ __forceinline__ void digits16(const double (&x0)[16], uint4 (&out)[S])
{
    double x[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) x[e] = x0[e];
#pragma unroll
    for (int p = 0; p < S; ++p) {
        uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
        for (int e = 0; e < 16; ++e) {
            const double d = rint(x[e]);
            x[e] = (x[e] - d) * 128.0; // exact: |x - rint(x)| <= 1/2
            w[e >> 2] |= ((uint32_t)(int)d & 0xFFu) << (8 * (e & 3));
        }
        out[p] = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

// T[i, ct] = K*[s0 + i, ct] - L[s0 + i, 0:s0] V[0:s0, ct] for one 128-row x 64-candidate tile; grid = nrows * n64, row tile fastest.
// Warp 0: TMA producer, warp 1: TMEM allocation + MMA issue, warps 2..5: epilogue (one row of L = one TMEM lane per thread).
__global__ void __launch_bounds__(THREADS, 1)
panel_update_i8_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const int* __restrict__ lexp,
    int ev, const double* __restrict__ V, int64_t ld, double* __restrict__ Tbuf, int64_t ldt, int s0, int nrows, int ct0,
    int* __restrict__ err)
{
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* full = (uint64_t*)(smem + (size_t)STAGES * STAGE_BYTES);
    uint64_t* empty = full + STAGES;
    uint64_t* tfull = empty + STAGES;
    uint32_t* tmem_base_s = (uint32_t*)(tfull + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int i = blockIdx.x % nrows, ct = ct0 + blockIdx.x / nrows;
    const int nk = s0 * LB_TILE / BK;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(tfull, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(lb_smem_u32(tmem_base_s)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_base_s;

    if (warp == 0) {
        if (lane == 0) { // ===== TMA producer =====
            int s = 0; uint32_t ph = 0;
            for (int kb = 0; kb < nk; ++kb) {
                if (!mbar_wait(&empty[s], ph ^ 1, err)) break;
                uint8_t* sa = smem + (size_t)s * STAGE_BYTES;
                mbar_expect_tx(&full[s], STAGE_BYTES);
                tma_load_3d(sa, &mapA, kb * BK, i * BM, &full[s]);
                tma_load_3d(sa + A_BYTES, &mapB, kb * BK, ct * BN, &full[s]);
                if (++s == STAGES) { s = 0; ph ^= 1; }
            }
        }
    }
    else if (warp == 1) {
        if (lane == 0) { // ===== MMA issuer: the 28 digit pairs i + j < S, pair (0, g) opens accumulator g =====
            int s = 0; uint32_t ph = 0; bool ok = true;
            for (int kb = 0; kb < nk; ++kb) {
                if (!mbar_wait(&full[s], ph, err)) { ok = false; break; }
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t sa = lb_smem_u32(smem + (size_t)s * STAGE_BYTES);
#pragma unroll
                for (int a = 0; a < S; ++a) {
                    const uint64_t adesc = desc_sw64(sa + a * A_PLANE);
#pragma unroll
                    for (int b = 0; a + b < S; ++b) {
                        const uint64_t bdesc = desc_sw64(sa + A_BYTES + b * B_PLANE);
#pragma unroll
                        for (int k = 0; k < BK / 32; ++k) // +32 B per MMA inside the 64 B swizzle row: +2 in the >>4 address field
                            umma_i8(tmem_base + (uint32_t)((a + b) * BN), adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k),
                                (kb | k | a) != 0);
                    }
                }
                umma_commit(&empty[s]);
                if (++s == STAGES) { s = 0; ph ^= 1; }
            }
            if (ok) umma_commit(tfull);
        }
    }
    else { // ===== epilogue: T = K* - 2^(e_r + e_V) sum_g 2^(-12 - 7 g) acc_g =====
        const int q = warp & 3;
        const int row = q * 32 + lane;
        if (mbar_wait_warp(tfull, 0, err)) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
            const int64_t grow = (int64_t)(s0 + i) * LB_TILE + row;
            const double scale = ldexp(1.0, lexp[grow] + ev);
            const double* kst = V + grow + (int64_t)ct * BN * ld;
            double* tout = Tbuf + (int64_t)i * LB_TILE + row + (int64_t)ct * BN * ldt;
#pragma unroll 1
            for (int c = 0; c < BN; c += 16) {
                double r[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) r[j] = 0.0;
#pragma unroll
                for (int g = S - 1; g >= 0; --g) {
                    uint32_t v[16];
                    tmem_ld16(taddr + (uint32_t)(g * BN + c), v);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                    const double w = ldexp(1.0, -12 - 7 * g);
#pragma unroll
                    for (int j = 0; j < 16; ++j) r[j] = fma((double)(int)v[j], w, r[j]);
                }
#pragma unroll
                for (int j = 0; j < 16; ++j) tout[(int64_t)(c + j) * ldt] = kst[(int64_t)(c + j) * ld] - scale * r[j];
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
    }
}

// lexp[r] = max over k < K(r) of the frexp exponent of L[r, k] (|L[r, k]| < 2^lexp[r]); grid (row tiles from 16 on, 256-column chunks)
__global__ void __launch_bounds__(256)
ldig_exp_kernel(const double* __restrict__ L, int64_t ld, int* __restrict__ lexp)
{
    __shared__ int red[256];
    const int t = 16 + blockIdx.x;                     // row tile
    const int64_t K = (int64_t)(t / 16) * SB_ROWS;      // k range of its super-block
    const int64_t k0 = (int64_t)blockIdx.y * 256;
    if (k0 >= K) return;
    const int row = threadIdx.x & 127, half = threadIdx.x >> 7;
    const int64_t r = (int64_t)t * LB_TILE + row;
    int e = INT_MIN;
    for (int64_t k = k0 + half; k < k0 + 256; k += 2) {
        const double v = L[r + k * ld];
        if (v != 0.0) e = max(e, ilogb(v) + 1);
    }
    red[threadIdx.x] = e;
    __syncthreads();
    if (half == 0) atomicMax(&lexp[r], max(e, red[threadIdx.x + 128]));
}

// digit planes of the super-block rectangles: plane p of super-block b (rows R_b = b * 2048 .., K_b = b * 2048) is row-major
// rows_b x K_b at dig + off_b + p * rows_b * K_b.  Tile of 64 rows x 64 k per CTA, transposed through shared memory.
__global__ void __launch_bounds__(256)
ldig_split_kernel(const double* __restrict__ L, int64_t ld, int64_t Np, const int* __restrict__ lexp, int8_t* __restrict__ dig)
{
    __shared__ double tile[64][65];
    const int64_t r0 = SB_ROWS + (int64_t)blockIdx.y * 64, k0 = (int64_t)blockIdx.x * 64;
    const int64_t b = r0 / SB_ROWS, K = b * SB_ROWS, R = b * SB_ROWS;
    if (k0 >= K) return;
    const int64_t rows = (Np - R < SB_ROWS) ? Np - R : SB_ROWS;
    const int64_t off = (int64_t)S * SB_ROWS * SB_ROWS * (b * (b - 1) / 2); // earlier super-blocks b' = 1 .. b-1: S x 2048 x b' 2048
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        const int idx = threadIdx.x + q * 256, rr = idx & 63, kk = idx >> 6;
        tile[kk][rr] = L[r0 + rr + (k0 + kk) * ld];
    }
    __syncthreads();
    const int rr = threadIdx.x >> 2, kq = (threadIdx.x & 3) * 16;
    const int e = lexp[r0 + rr];
    double x[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) x[j] = ldexp(tile[kq + j][rr], 6 - e);
    uint4 d[S];
    digits16(x, d);
    int8_t* base = dig + off + (r0 + rr - R) * K + k0 + kq;
#pragma unroll
    for (int p = 0; p < S; ++p) *reinterpret_cast<uint4*>(base + (int64_t)p * rows * K) = d[p];
}

// digit planes of V rows [r0, r0 + nr) x columns [c0, c0 + nc): plane p at vdig + p * Np * Mp, same layout as V (k contiguous)
__global__ void __launch_bounds__(256)
vdig_split_kernel(const double* __restrict__ V, int64_t ld, int64_t Mp, int64_t r0, int64_t nr, int64_t c0, int64_t nc, int ev,
    int8_t* __restrict__ vdig)
{
    const int64_t per_col = nr / 16;
    const int64_t idx = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (idx >= per_col * nc) return;
    const int64_t c = c0 + idx / per_col, r = r0 + (idx % per_col) * 16;
    const double* src = V + r + c * ld;
    double x[16];
#pragma unroll
    for (int j = 0; j < 16; j += 2) {
        const double2 v2 = *reinterpret_cast<const double2*>(src + j);
        x[j] = ldexp(v2.x, 6 - ev);
        x[j + 1] = ldexp(v2.y, 6 - ev);
    }
    uint4 d[S];
    digits16(x, d);
    int8_t* dst = vdig + r + c * ld;
#pragma unroll
    for (int p = 0; p < S; ++p) *reinterpret_cast<uint4*>(dst + (int64_t)p * ld * Mp) = d[p];
}

// 3-D uint8 tensor map: {k (inner, K bytes), rows, S planes}, boxes of {64, box_rows, S}, 64-byte swizzle
int make_map(CUtensorMap* map, const void* base, int64_t K, int64_t rows, int64_t row_stride, int64_t plane_stride, int box_rows)
{
    EncodeTiledFn enc = get_encode();
    if (!enc) return LB_ERR_UNSUPPORTED;
    cuuint64_t gdim[3] = {(cuuint64_t)K, (cuuint64_t)rows, (cuuint64_t)S};
    cuuint64_t gstr[2] = {(cuuint64_t)row_stride, (cuuint64_t)plane_stride};
    cuuint32_t box[3] = {(cuuint32_t)BK, (cuuint32_t)box_rows, (cuuint32_t)S};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, (void*)base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
        CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? LB_OK : LB_ERR_CUDA;
}

int64_t ldig_plane_bytes(int64_t Np)
{
    int64_t total = 0;
    for (int64_t R = SB_ROWS; R < Np; R += SB_ROWS) total += (int64_t)S * ((Np - R < SB_ROWS) ? Np - R : SB_ROWS) * R;
    return total;
}
// offset of super-block b >= 1 (every earlier super-block has all 2048 rows)
int64_t ldig_offset(int64_t b) { return (int64_t)S * SB_ROWS * SB_ROWS * (b * (b - 1) / 2); }

LbOncePerDevice g_attr_once;
int g_mode = -1;         // 1: int8 update (default), 0: DMMA update
int64_t g_max_k = -1;    // longest K range taken by the int8 kernel

} // namespace qi8

// LB_QUERY_INT8=0 restores the DMMA update of the panel query
int lb_query_int8_mode()
{
    if (qi8::g_mode < 0) {
        const char* e = getenv("LB_QUERY_INT8");
        qi8::g_mode = (e && atoi(e) == 0) ? 0 : 1;
    }
    return qi8::g_mode;
}
int64_t lb_query_int8_max_k() { return qi8::g_max_k > 0 ? qi8::g_max_k : qi8::MAX_K; }

// testing hook: on = 1 / 0 selects the int8 / DMMA update (< 0: LB_QUERY_INT8 again); max_k > 0 lowers the K bound of the int8
// kernel (super-blocks beyond it take the DMMA update), <= 0 restores the exactness bound
extern "C" int lb_debug_set_query_int8(int on, long long max_k)
{
    qi8::g_mode = on < 0 ? -1 : (on != 0);
    qi8::g_max_k = (max_k > 0 && max_k <= qi8::MAX_K) ? (int64_t)max_k : -1;
    return LB_OK;
}

size_t lb_query_i8_vdig_bytes(int64_t Np, int64_t Mp) { return (size_t)qi8::S * (size_t)Np * (size_t)Mp; }

// Digit planes and row exponents of L for the panel query, kept until the next factorisation (h->ldig_valid).
int lb_ldig_prepare(lb_gp* h)
{
    using namespace qi8;
    if (h->ldig_valid) return LB_OK;
    const int64_t Np = h->Np, T = Np / LB_TILE;
    const size_t planes = (size_t)ldig_plane_bytes(Np);
    const size_t bytes = planes + sizeof(int) * (size_t)Np;
    if (!h->dLdig || h->ldig_np != Np || lb_pool_shared(h->dLdig)) { // a clone's planes are never overwritten
        lb_dfree_sync(h, h->dLdig);
        h->dLdig = nullptr;
        LB_ALLOC(h, h->dLdig, bytes);
        h->ldig_np = Np;
    }
    if (T > SB_ROWS / LB_TILE) {
        int* lexp = reinterpret_cast<int*>(h->dLdig + planes);
        LB_CUDA(cudaMemsetAsync(lexp, 0x80, sizeof(int) * (size_t)Np, h->stream));
        const int64_t kmax = (T - 1) / 16 * SB_ROWS; // K range of the last super-block
        ldig_exp_kernel<<<dim3((unsigned)(T - 16), (unsigned)(kmax / 256)), 256, 0, h->stream>>>(h->dL, Np, lexp);
        ldig_split_kernel<<<dim3((unsigned)(kmax / 64), (unsigned)((Np - SB_ROWS) / 64)), 256, 0, h->stream>>>(h->dL, Np, Np, lexp, h->dLdig);
        h->launches += 2;
        LB_CUDA(cudaGetLastError());
    }
    h->ldig_valid = true;
    return LB_OK;
}

// frexp exponent of sigma_f: |V| <= sigma_f < 2^e
int lb_query_i8_vexp(const lb_gp* h) { return std::ilogb(std::sqrt(h->kp.sf2)) + 1; }

int lb_launch_vdig_split(cudaStream_t st, const double* dV, int64_t ld, int64_t Mp, int64_t r0, int64_t nr, int64_t c0, int64_t nc, int ev,
    int8_t* dVdig)
{
    const int64_t n = nr / 16 * nc;
    qi8::vdig_split_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dV, ld, Mp, r0, nr, c0, nc, ev, dVdig);
    LB_CUDA(cudaGetLastError());
    return LB_OK;
}

// Tbuf tiles of super-block s0 (nrows row tiles) for the 64-wide candidate tiles [ct0, ct0 + n64).  K = s0 * 128 <= lb_query_int8_max_k().
int lb_launch_panel_update_i8(const lb_gp* h, cudaStream_t st, const double* dV, const int8_t* dVdig, int64_t Mp, double* dT, int64_t ldt,
    int s0, int nrows, int ct0, int n64, int ev, int* dErr)
{
    using namespace qi8;
    const int64_t Np = h->Np, K = (int64_t)s0 * LB_TILE;
    if (s0 <= 0 || s0 % (SB_ROWS / LB_TILE) || K > lb_query_int8_max_k() || !h->ldig_valid) return LB_ERR_ARG;
    if (g_attr_once.need()) LB_CUDA(cudaFuncSetAttribute(panel_update_i8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
    const int64_t rows_b = (Np - K < SB_ROWS) ? Np - K : SB_ROWS;
    const int8_t* dA = h->dLdig + ldig_offset(K / SB_ROWS);
    const int* lexp = reinterpret_cast<const int*>(h->dLdig + ldig_plane_bytes(Np));
    alignas(64) CUtensorMap mapA, mapB;
    int rc;
    if ((rc = make_map(&mapA, dA, K, rows_b, K, rows_b * K, BM))) return rc;
    if ((rc = make_map(&mapB, dVdig, Np, Mp, Np, Np * Mp, BN))) return rc;
    panel_update_i8_kernel<<<(unsigned)(nrows * n64), THREADS, SMEM_BYTES, st>>>(mapA, mapB, lexp, ev, dV, Np, dT, ldt, s0, nrows, ct0, dErr);
    LB_CUDA(cudaGetLastError());
    return LB_OK;
}
