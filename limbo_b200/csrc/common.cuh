// limbo_b200/csrc/common.cuh — shared declarations for the sm_100a GP backend.
//
// Data layout in HBM (see DESIGN.md §3):
//   * every N-sized dimension is padded to Np = roundup(N, 128); the padded
//     part of K is the identity, so the Cholesky factor, the triangular
//     solves, K^-1 and log|K| of the padded system restrict exactly to those
//     of the N x N system and no kernel needs edge predication;
//   * X  : D x Np "SoA" (dimension-major) so 128-point blocks of one input
//     dimension are 1 KB contiguous runs (TMA bulk-copy friendly);
//   * K/L: Np x Np column-major (Eigen::MatrixXd's layout, gp.hpp:553), the
//     factor overwrites the lower triangle in place;
//   * invD: T blocks of 128 x 128 (column-major, lower) = inverses of the
//     diagonal blocks of L, produced by the panel factorisation and reused by
//     every triangular solve.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>

#define LB_TILE 128
#define LB_NEV 8 // events per handle: fork / panel x2 / a-update x2 / join / second-group fork + join

// ---- status codes (include/limbo_b200.h) ----------------------------------
#define LB_OK 0
#define LB_ERR_ARG (-1)
#define LB_ERR_CUDA (-2)
#define LB_ERR_STATE (-3)
#define LB_ERR_ALLOC (-4)
#define LB_ERR_UNSUPPORTED (-5)
#define LB_ERR_TIMEOUT (-6)

#define LB_CUDA(call)                                                                   \
    do {                                                                                \
        cudaError_t e__ = (call);                                                       \
        if (e__ != cudaSuccess) {                                                       \
            lb_set_last_cuda_error(e__, __FILE__, __LINE__);                            \
            return LB_ERR_CUDA;                                                         \
        }                                                                               \
    } while (0)

void lb_set_last_cuda_error(cudaError_t e, const char* file, int line);

enum { LB_K_SE_ARD = 0, LB_K_MATERN52 = 1, LB_K_MATERN32 = 2, LB_K_EXP = 3 };
#define LB_MAX_D 64
#define LB_MAX_LAMBDA 4 // columns of the SE-ARD Lambda matrix (Params::kernel_squared_exp_ard::k)
#define LB_MAX_HPARAMS (LB_MAX_D * (1 + LB_MAX_LAMBDA) + 2) // SE-ARD: log ell, Lambda columns, log sigma_f, (noise)

// Kernel parameters passed by value to device code.
struct KernParams {
    int id;
    int D;
    double sf2;      // exp(2 p_last)                    squared_exp_ard.hpp:104
    double l;        // isotropic length scale            matern_five_halves.hpp:100
    double noise;    // kernel/kernel.hpp:76-79
    double inv_ell[LB_MAX_D]; // SE-ARD: 1/exp(p_d)
    double c1;       // Matern: sqrt(5)/l resp. sqrt(3)/l ; Exp: 1/l^2   (host-precomputed, saves a divide per pair)
    double c2;       // Matern-5/2: 5/(3 l^2)
    // SE-ARD with k > 0 (squared_exp_ard.hpp:109-126,142-146): z = d^T (A A^T + diag(ell^-2)) d = |W^T d|^2 with
    // W = [diag(1/ell) | A].  The staged samples carry D = Draw + klam coordinates (x/ell, A^T x), so every kernel that
    // consumes the staged tiles is unchanged; only the staging and the gradient wrt A know about A.
    int Draw;        // input dimension of the caller's points
    int klam;        // number of columns of A
    const double* lambda; // device, Draw x klam column-major (nullptr when klam == 0)
};

// ---------------------------------------------------------------------------
// Device-side kernel functor: value from the (scaled) squared distance.
//   SE-ARD : z = sum_d ((x_d - y_d)/ell_d)^2  (X is pre-scaled by 1/ell_d)
//   others : z = sum_d (x_d - y_d)^2          (raw X)
// Operation order after z follows the reference functors so that the result
// differs from the Eigen path only by the rounding of z itself.
// ---------------------------------------------------------------------------
__device__ __forceinline__ double lb_kernel_from_z(int id, double z, double sf2, double l)
{
    switch (id) {
    case LB_K_SE_ARD: // squared_exp_ard.hpp:150
        return sf2 * exp(-0.5 * z);
    case LB_K_MATERN52: { // matern_five_halves.hpp:104-113
        double d = sqrt(z);
        double d_sq = d * d;
        double l_sq = l * l;
        double term1 = sqrt(5.0) * d / l;
        double term2 = 5. * d_sq / (3. * l_sq);
        return sf2 * (1 + term1 + term2) * exp(-term1);
    }
    case LB_K_MATERN32: { // matern_three_halves.hpp:102-108
        double d = sqrt(z);
        double term = sqrt(3.0) * d / l;
        return sf2 * (1 + term) * exp(-term);
    }
    default: { // exp.hpp:94-99
        double r = z / (l * l);
        return sf2 * exp(-0.5 * r);
    }
    }
}

// exp(t) for t <= 0, branch-free: n = rint(t log2 e), r = t - n ln 2 (two-term), degree-13 Taylor in |r| <= 0.347
// (truncation < 5e-18), 2^n by an exponent-field add.  Relative error < 3e-16 for t >= -708 (tests/test_gpu_tf32.py),
// exactly 0 below (where the reference's std::exp returns a denormal < 2.3e-308).  ~18 fp64 instructions and no slow-path
// branch, so the 32 evaluations a thread holds interleave: the kernel-evaluation loops (K build, K*, gradient) are bound
// by the fp64 pipe whenever they are not bound by HBM.
__device__ __forceinline__ double lb_exp_nonpos(double t)
{
    const double MAGIC = 6755399441055744.0; // 1.5 * 2^52
    double fn = fma(t, 1.4426950408889634074, MAGIC);
    const int n = __double2loint(fn);
    fn -= MAGIC;
    double r = fma(fn, -6.93147180369123816490e-01, t);
    r = fma(fn, -1.90821492927058770002e-10, r);
    double p = 1.6059043836821614599e-10; // 1/13!
    p = fma(p, r, 2.0876756987868098979e-09);
    p = fma(p, r, 2.5052108385441718775e-08);
    p = fma(p, r, 2.7557319223985890653e-07);
    p = fma(p, r, 2.7557319223985890653e-06);
    p = fma(p, r, 2.4801587301587301587e-05);
    p = fma(p, r, 1.9841269841269841270e-04);
    p = fma(p, r, 1.3888888888888888889e-03);
    p = fma(p, r, 8.3333333333333333333e-03);
    p = fma(p, r, 4.1666666666666666667e-02);
    p = fma(p, r, 1.6666666666666666667e-01);
    p = fma(p, r, 0.5);
    p = fma(p, r, 1.0);
    p = fma(p, r, 1.0);
    const int hi = __double2hiint(p) + (n << 20);
    const double e = __hiloint2double(hi, __double2loint(p));
    return t < -708.0 ? 0.0 : e;
}

// Same functors with the per-pair divisions and the square root replaced by host-precomputed reciprocals and a
// branch-free rsqrt (<= a few ulp from the reference's operation order; K stays within 1e-15 of the Eigen path).
__device__ __forceinline__ double lb_rsqrt_nr(double x)
{
    double r;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    const double h = 0.5 * x;
    r = fma(r, fma(-h * r, r, 0.5), r);
    r = fma(r, fma(-h * r, r, 0.5), r);
    return r;
}
__device__ __forceinline__ double lb_kernel_from_z(int id, double z, const KernParams& kp)
{
    switch (id) {
    case LB_K_SE_ARD:
        return kp.sf2 * exp(-0.5 * z); // libm here: the SE-ARD K build is HBM bound with it (0.85 of peak) and compute bound (0.67) with lb_exp_nonpos
    case LB_K_MATERN52: {
        // sigma_f^2 (1 + c1 d + c2 d^2) exp(-c1 d) with d^2 = z and sigma_f^2 folded into the polynomial (two FMAs instead of
        // two products and two sums; <= 2 ulp from the reference's operation order, matern_five_halves.hpp:106-112): the
        // Matern K build is bound by the fp64 pipe, not by HBM (~45 fp64 instructions per element)
        const double d = (z > 0.0) ? z * lb_rsqrt_nr(z) : 0.0;
        const double term1 = kp.c1 * d;
        return fma(kp.c2 * kp.sf2, z, fma(kp.sf2, term1, kp.sf2)) * lb_exp_nonpos(-term1);
    }
    case LB_K_MATERN32: {
        const double d = (z > 0.0) ? z * lb_rsqrt_nr(z) : 0.0;
        const double term = kp.c1 * d;
        return fma(kp.sf2, term, kp.sf2) * lb_exp_nonpos(-term);
    }
    default:
        return kp.sf2 * exp(-0.5 * (z * kp.c1));
    }
}

// Normalised kernel value (sigma_f^2 = 1) from the (scaled) squared distance, kernel id as a template parameter.
template <int KID>
__device__ __forceinline__ double lb_unit_kernel_from_z(double z, const KernParams& kp)
{
    if (KID == LB_K_SE_ARD) return lb_exp_nonpos(-0.5 * z);
    if (KID == LB_K_MATERN52) {
        const double d = (z > 0.0) ? z * lb_rsqrt_nr(z) : 0.0;
        const double term1 = kp.c1 * d;
        return (1 + term1 + kp.c2 * (d * d)) * lb_exp_nonpos(-term1);
    }
    if (KID == LB_K_MATERN32) {
        const double d = (z > 0.0) ? z * lb_rsqrt_nr(z) : 0.0;
        const double term = kp.c1 * d;
        return (1 + term) * lb_exp_nonpos(-term);
    }
    return lb_exp_nonpos(-0.5 * (z * kp.c1));
}

// staged coordinate d (0 <= d < kp.D) of a raw point given by x(r), r < kp.Draw
template <typename F>
__device__ __forceinline__ double lb_staged_coord(const KernParams& kp, int d, F&& x)
{
    if (kp.id != LB_K_SE_ARD) return x(d);
    if (d < kp.Draw) return x(d) * kp.inv_ell[d]; // squared_exp_ard.hpp:148: cwiseQuotient(_ell), applied once per point
    double s = 0.0;
    const double* a = kp.lambda + (int64_t)(d - kp.Draw) * kp.Draw;
    for (int r = 0; r < kp.Draw; ++r) s = fma(a[r], x(r), s);
    return s;
}

// ---------------------------------------------------------------------------
// PTX helpers
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t lb_smem_u32(const void* p)
{
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// fp64 tensor-core MMA (DMMA).  tcgen05 has no f64 kind; on sm_100a the fp64
// tensor path is warp-level mma.sync, which ptxas lowers to DMMA.8x8x4.
//   A frag (16x8, row): a[i]: row = g + 8*(i&1), col = t + 4*(i>>1)
//   B frag (8x8,  col): b[i]: k = t + 4*i, n = g
//   C frag (16x8)     : c[i]: row = g + 8*(i>>1), col = 2*t + (i&1)
// with g = lane>>2, t = lane&3.
__device__ __forceinline__ void lb_dmma_16x8x8(double (&c)[4], const double (&a)[4], const double (&b)[2])
{
    asm volatile(
        "mma.sync.aligned.m16n8k8.row.col.f64.f64.f64.f64 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
        : "+d"(c[0]), "+d"(c[1]), "+d"(c[2]), "+d"(c[3])
        : "d"(a[0]), "d"(a[1]), "d"(a[2]), "d"(a[3]), "d"(b[0]), "d"(b[1]));
}

// The native SASS shape.  ptxas lowers one m16n8k8 into FOUR chained DMMA.8x8x4 (k0-3 -> temp -> k4-7 per row
// half), i.e. no instruction-level parallelism inside a warp; issuing m8n8k4 ourselves, one independent tile after
// the other, keeps dependent DMMAs a whole tile-sweep apart.
//   a: A[row g][k t]   b: B[k t][n g]   c0,c1: C[row g][cols 2t, 2t+1]
__device__ __forceinline__ void lb_dmma_8x8x4(double& c0, double& c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

__device__ __forceinline__ void lb_cp_async16(void* smem_dst, const void* gmem_src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(lb_smem_u32(smem_dst)), "l"(gmem_src));
}
__device__ __forceinline__ void lb_cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void lb_cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// mbarrier + TMA 1-D bulk copy (cp.async.bulk -> SASS UBLKCP)
__device__ __forceinline__ void lb_mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(lb_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void lb_fence_barrier_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::);
}
__device__ __forceinline__ void lb_fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;\n" ::);
}
__device__ __forceinline__ void lb_mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(lb_smem_u32(bar)), "r"(bytes));
}
__device__ __forceinline__ void lb_mbar_wait(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}\n" ::"r"(lb_smem_u32(bar)),
        "r"(parity));
}
// bytes must be a multiple of 16; src/dst 16-byte aligned
__device__ __forceinline__ void lb_bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                     lb_smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(lb_smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ double lb_warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---------------------------------------------------------------------------
// Host-side handle
// ---------------------------------------------------------------------------
struct lb_gp {
    int device = 0;
    int precision = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaStream_t side = nullptr;   // high-priority stream for the look-ahead panel factorisation
    cudaStream_t aux = nullptr;    // normal-priority second stream (panel query: second column group), created on first use
    cudaStream_t aux2 = nullptr, aux3 = nullptr; // third / fourth column group of the panel query for small batches (created on first use)
    cudaEvent_t ev[LB_NEV] = {};        // fork / panel / a-update / join events

    int64_t N = 0;   // live samples
    int64_t Np = 0;  // padded capacity (multiple of 128)
    int D = 0, P = 0;

    KernParams kp{};
    bool kernel_set = false;
    int n_hparams = 0;

    double* dX = nullptr;    // D x Np raw samples (SoA)
    double* dXs = nullptr;   // (D + LB_MAX_LAMBDA) x Np samples staged for the kernel (SE-ARD: x/ell, then A^T x)
    double* dLambda = nullptr; // D x LB_MAX_LAMBDA (SE-ARD A matrix)
    double* dLinvW = nullptr; int64_t linvw_np = 0; // reduced-precision path: |L^-1 e_k|^2 per column (rounding-bias weights)
    double* dY = nullptr;    // Np x P  obs_mean (col-major), zero padded
    double* dL = nullptr;    // Np x Np K then L (col-major)
    double* dInvD = nullptr; // T x 128 x 128
    double* dAlpha = nullptr; // Np x P
    double* dLinv = nullptr; // Np x Np (lazy: L^-1)
    double* dKinv = nullptr; // Np x Np (lazy: K^-1, lower valid + mirrored)
    int8_t* dLdig = nullptr; int64_t ldig_np = 0; bool ldig_valid = false; // panel query: int8 digit planes of L (query_i8.cu)
    float* dLinv32 = nullptr; int64_t linv32_rows = 0; bool linv32_valid = false; double linv32_scale = 1.0; // reduced-precision path: row-major fp32 / fp16 L^-1
    int* dInfo = nullptr;    // [0] first failing pivot (1-based) or 0; [1] solver error
    int* dFlags = nullptr;   // T+8 ints: ticket counters of the persistent solves
    double* dTrsvX = nullptr; int64_t trsvx_np = 0; // trsv: published solution blocks (sentinel-filled per launch)
    double* dScratch = nullptr; size_t scratch_bytes = 0;

    bool fitted = false;
    bool linv_valid = false;
    int linv_levels = 0;     // diagonal blocks of this many 128-tiles of dLinv hold the inverse (0: nothing, >= T: all of L^-1)
    bool kinv_valid = false;
    bool kinv_sym = false;   // upper triangle of dKinv mirrored (needed by the LOO products and lb_get)
    double* dWork = nullptr; int64_t work_np = 0; // Np x Np workspace (dK/dtheta of the LOO gradient)
    bool force_unfused = false; // tests: use the multi-launch query path

    // counters for bench.py ("gpu_launches")
    long long launches = 0;
    void* prof = nullptr; // Profiler* when per-kernel-class event timing is enabled (abi.cu)
};

// Every extern "C" entry that takes a handle runs on the handle's device and restores the caller's current device on
// return (one process may hold handles on several GPUs, e.g. one MultiGP output per device).
struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(const lb_gp* h)
    {
        if (!h) return;
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != h->device && cudaSetDevice(h->device) != cudaSuccess) ok = false;
    }
    ~DeviceGuard()
    {
        if (prev >= 0) {
            int cur = -1;
            if (cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
        }
    }
};
#define LB_DEVICE(h)                        \
    DeviceGuard lb_dev_guard__(h);          \
    if (!lb_dev_guard__.ok) return LB_ERR_CUDA

// cudaFuncSetAttribute applies to the CURRENT device: once-only flags must be per device (one process may hold handles on
// several GPUs, e.g. one MultiGP output per device).  need() is true the first time it is called on a device.
struct LbOncePerDevice {
    bool done[64] = {};
    bool need()
    {
        int d = 0;
        if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= 64) return true;
        if (done[d]) return false;
        done[d] = true;
        return true;
    }
};

// pooled, reference-counted device buffers (pool.cu): every buffer a handle owns comes from here
void* lb_pool_alloc(int device, size_t bytes);
void lb_pool_free(void* p);     // drops one reference; the buffer returns to the pool with the last one
void lb_pool_retain(void* p);
bool lb_pool_shared(void* p);   // more than one handle references the buffer
template <typename T>
inline int lb_dalloc(const lb_gp* h, T** p, size_t bytes)
{
    *p = static_cast<T*>(lb_pool_alloc(h->device, bytes));
    return *p ? LB_OK : LB_ERR_ALLOC;
}
// cudaFree synchronises implicitly, the pool does not: wait for the handle's pending work before a buffer that
// kernels in flight may still use goes back to the pool
template <typename H>
inline void lb_dfree_sync(H* h, void* p)
{
    if (!p) return;
    cudaStreamSynchronize(h->stream);
    lb_pool_free(p);
}
#define LB_ALLOC(h, ptr, bytes)                      \
    do {                                             \
        int rc_alloc__ = lb_dalloc((h), &(ptr), (bytes)); \
        if (rc_alloc__) return rc_alloc__;           \
    } while (0)

// per-kernel-class CUDA-event timing (bench.py roofline): no-ops unless enabled
enum { LB_PC_KBUILD = 0, LB_PC_POTF2, LB_PC_TRSM_PANEL, LB_PC_SYRK, LB_PC_SYRK_COL, LB_PC_TRSV, LB_PC_KSTAR, LB_PC_QSTEP, LB_PC_QREDUCE,
    LB_PC_ACQ, LB_PC_TRTRI, LB_PC_LAUUM, LB_PC_GRAD, LB_PC_OTHER, LB_PC_COUNT };
void lb_prof_begin(const lb_gp* h, cudaStream_t st, int cls);
void lb_prof_end(const lb_gp* h, cudaStream_t st, int cls);
struct LbProfScope {
    const lb_gp* h; cudaStream_t st; int cls;
    LbProfScope(const lb_gp* h_, cudaStream_t st_, int c) : h(h_), st(st_), cls(c) { if (h->prof) lb_prof_begin(h, st, cls); }
    ~LbProfScope() { if (h->prof) lb_prof_end(h, st, cls); }
};

// internal entry points (one per .cu)
int lb_launch_scale_x(lb_gp* h);
int lb_launch_kbuild(lb_gp* h, double* dK);
int lb_launch_potrf(lb_gp* h);
int lb_launch_solve_alpha(lb_gp* h);
int lb_launch_trsv(lb_gp* h, double* dB, int nrhs, bool forward);
int lb_launch_query(const lb_gp* h, cudaStream_t st, int64_t M, const double* dXq_soa /*D x Mp*/, int64_t Mp,
    double* dV /*Np x Mp*/, double* dMu /*Mp x P*/, double* dS2 /*Mp*/, long long* launches);
int lb_launch_acq(const lb_gp* h, cudaStream_t st, int acq_id, double p0, double p1, int64_t M, const double* dMu0,
    const double* dS2, double* dAcq, double* dBestVal, long long* dBestIdx, long long* launches);
int lb_launch_loglik(lb_gp* h, double* dOut /*3 doubles: a, logdet, loglik*/);
int lb_launch_kinv(lb_gp* h);
int lb_launch_linv_levels(lb_gp* h, int want_tiles); // lml.cu: inverse of the diagonal blocks of `want_tiles` 128-tiles (power of two)
int lb_launch_grad(lb_gp* h, int optimize_noise, double* dGrad);
int lb_ensure_scratch(lb_gp* h, size_t bytes);
int lb_query_int8_mode(); // query_i8.cu: int8 digit-product update of the panel query (LB_QUERY_INT8)
int lb_tf32_prepare(lb_gp* h);
int lb_launch_tf32_gemm_norm(cudaStream_t st, const void* dA, int64_t lda, const void* dB, int64_t ldb, int64_t M, int64_t N, int64_t K,
    int tri, float* dNorm2, float* dDout, int* dErr, int grid, int f16);
int lb_launch_tf32_gemm_norm_cluster(cudaStream_t st, const void* dA, int64_t lda, const void* dB, int64_t ldb, int64_t M, int64_t N,
    int64_t K, int tri, float* dNorm2, int* dErr, int sms, int cl, int f16);
int lb_tf32_cluster_size();
int lb_launch_kstar_tf32(const lb_gp* h, cudaStream_t st, int64_t Mc, const double* dQs, int64_t Mcp, float* dKt, double* dMuPart,
    double* dMu, double* dBias, long long* launches);
int lb_launch_sigma_tf32(const lb_gp* h, cudaStream_t st, int64_t Mc, int64_t Mcp, const float* dKt, float* dNorm2, int* dErr,
    const double* dBias, double* dS2, long long* launches);
