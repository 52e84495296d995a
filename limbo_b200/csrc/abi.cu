// limbo_b200/csrc/abi.cu — extern "C" boundary (include/limbo_b200.h) and the
// host-side orchestration of the device pipeline.  No torch types, no CPU
// fallback: every numerical result below comes from the CUDA kernels in this
// directory.
#include "../../include/limbo_b200.h"
#include "common.cuh"
#include <algorithm>
#include <cmath>
#include <cstring>
#include <cstdio>
#include <mutex>
#include <new>
#include <string>

int lb_launch_potf2_block(lb_gp* h, int k, int do_factor);
int lb_debug_potf2_clocks(lb_gp* h, int k, long long* out_host, int n);
int lb_launch_linv(lb_gp* h);
int lb_launch_symmetrize(lb_gp* h, double* dA);
int lb_launch_loo_value(lb_gp* h, double* dOut);
int lb_launch_loo_grad(lb_gp* h, int optimize_noise, double* dGrad);
int lb_launch_kinv_obs(lb_gp* h, double* dOut);
int lb_query_fused_supported(const lb_gp* h);
size_t lb_query_panel_scratch_doubles(const lb_gp* h, int64_t Mp);
size_t lb_linv_columns_scratch_doubles(const lb_gp* h, int G);
int lb_launch_linv_columns(lb_gp* h, cudaStream_t st, int rank, int G, double* dWork, long long* launches);
size_t lb_dinv_chunk_bytes_impl(const lb_gp* h, int G);
int lb_dinv_absmax(lb_gp* h, const double* dV, int G, double* out);
int lb_dinv_pack_impl(lb_gp* h, const double* dV, int rank, int G, double absmax_all, void* dChunk);
int lb_dinv_adopt_impl(lb_gp* h, int G, const void* dAll, double absmax_all);
int lb_launch_query_point(const lb_gp* h, cudaStream_t st, const double* x_host, double* dQs, double* dVscratch, double* dOutMapped,
    long long* launches);
int lb_launch_query_panel(lb_gp* h, cudaStream_t st, int64_t M, const double* dQs, int64_t Mp, double* dWork, double* dMu, double* dS2, int* dErr,
    long long* launches);
size_t lb_query_fused_scratch_doubles(const lb_gp* h, int grid);
int lb_launch_query_fused(const lb_gp* h, cudaStream_t st, int64_t M, const double* dQs, int64_t Mp, double* dVscratch,
    int grid, double* dMu, double* dS2, long long* launches);
int lb_launch_acq_full(cudaStream_t st, int acq_id, double p0, double p1, int64_t M, const double* dMu, int mu_stride,
    const double* dMeanAtQ, double mean_const, const double* dS2, double* dAcq, double* dBlkVal, long long* dBlkIdx,
    double* dBestVal, long long* dBestIdx, long long* launches);

static thread_local std::string g_last_cuda_error;
void lb_set_last_cuda_error(cudaError_t e, const char* file, int line)
{
    char buf[512];
    snprintf(buf, sizeof(buf), "%s (%s) at %s:%d", cudaGetErrorName(e), cudaGetErrorString(e), file, line);
    g_last_cuda_error = buf;
    cudaGetLastError(); // clear sticky-less errors
}

#include <vector>
struct Profiler {
    struct Rec { cudaEvent_t a, b; int cls; };
    std::vector<Rec> recs;
    std::vector<cudaEvent_t> pool;
    cudaEvent_t cur[LB_PC_COUNT] = {};
    double ms[LB_PC_COUNT] = {};
    long long n[LB_PC_COUNT] = {};
    std::mutex mu;
    cudaEvent_t get()
    {
        if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
        cudaEvent_t e; cudaEventCreate(&e); return e;
    }
};
void lb_prof_begin(const lb_gp* h, cudaStream_t st, int cls)
{
    Profiler* p = (Profiler*)h->prof;
    std::lock_guard<std::mutex> lk(p->mu);
    cudaEvent_t e = p->get();
    cudaEventRecord(e, st);
    p->cur[cls] = e;
}
void lb_prof_end(const lb_gp* h, cudaStream_t st, int cls)
{
    Profiler* p = (Profiler*)h->prof;
    std::lock_guard<std::mutex> lk(p->mu);
    cudaEvent_t e = p->get();
    cudaEventRecord(e, st);
    p->recs.push_back({p->cur[cls], e, cls});
}

namespace {

struct QueryWs { // per-handle query workspace (guarded by qmutex)
    double* dQraw = nullptr; size_t qraw_bytes = 0;   // M x D row-major staging
    double* dQs = nullptr; size_t qs_bytes = 0;       // D x Mp
    double* dV = nullptr; size_t v_bytes = 0;         // Np x Mc
    double* dMu = nullptr; size_t mu_bytes = 0;       // M x P
    double* dS2 = nullptr; size_t s2_bytes = 0;       // M
    double* dAcq = nullptr; size_t acq_bytes = 0;     // M
    double* dBlkVal = nullptr; long long* dBlkIdx = nullptr; size_t blk_cap = 0;
    double* dBest = nullptr; // [0] value ; long long index follows
    long long* dBestIdx = nullptr;
    double* dMean = nullptr; size_t mean_bytes = 0;
    float* dKt = nullptr; size_t kt_bytes = 0;         // TF32 path: K*^T chunk (Mc x Np fp32)
    float* dNorm2 = nullptr; size_t norm2_bytes = 0;
    double* dBias = nullptr; size_t bias_bytes = 0;    // reduced-precision path: rounding-bias weight per candidate
    int* dErr = nullptr;
};

struct Extra {
    std::mutex qmutex;
    QueryWs ws;
    double* dMisc = nullptr; // small scalars (loglik outputs, grad)
    cudaStream_t own = nullptr; // the handle's own stream (h->stream may point at a caller's stream)
    double lambda_host[LB_MAX_D * LB_MAX_LAMBDA] = {}; // host mirror of dLambda (lb_set_kernel compares against it)
    long long n_append = 0; // incremental updates actually taken (tests)
    double* hPoint = nullptr;  // pinned, mapped host buffer for the one-point query (mu[P], sigma^2)
    double* dPoint = nullptr;  // its device alias
    int point_cap = 0;
};

} // namespace

// The Extra block is stored behind the public struct.
struct lb_gp_full : lb_gp {
    Extra ex;
};
static inline lb_gp_full* full(const lb_gp* h) { return static_cast<lb_gp_full*>(const_cast<lb_gp*>(h)); }

namespace {

template <typename T>
int ensure(const lb_gp* h, T** p, size_t* cap, size_t bytes)
{
    if (*cap >= bytes && *p) return LB_OK;
    lb_dfree_sync(h, *p); // kernels in flight may still use the old buffer
    *p = nullptr;
    *cap = 0;
    const size_t want = bytes + 256;
    int rc = lb_dalloc(h, p, want);
    if (rc) return rc;
    *cap = want;
    return LB_OK;
}

// Make *p private to h before h writes it (copy-on-write for buffers lb_clone shares).  preserve = keep the contents;
// otherwise the caller overwrites the whole buffer and the copy is skipped.  A missing buffer is allocated.
template <typename T>
int make_unique(lb_gp* h, T** p, size_t bytes, bool preserve, bool* fresh = nullptr)
{
    if (fresh) *fresh = false;
    if (*p && !lb_pool_shared(*p)) return LB_OK;
    T* n = nullptr;
    LB_ALLOC(h, n, bytes);
    if (fresh) *fresh = true;
    if (*p) {
        if (preserve) {
            LB_CUDA(cudaMemcpyAsync(n, *p, bytes, cudaMemcpyDeviceToDevice, h->stream));
            LB_CUDA(cudaStreamSynchronize(h->stream)); // the other holder may write the buffer once it is its sole owner
        }
        lb_pool_free(*p);
    }
    *p = n;
    return LB_OK;
}

// row-major (n x D) -> dimension-major (D x np) with optional per-dimension scale, zero padded
__global__ void pack_soa_kernel(const double* __restrict__ src, int64_t n, int D, double* __restrict__ dst, int64_t np,
    KernParams kp, int scaled)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    int d = blockIdx.y;
    if (i >= np) return;
    // D = row length of src; grid.y = D (raw copy) or kp.D (staged for the kernel: x/ell and the Lambda projections)
    double v = 0.0;
    if (i < n) v = scaled ? lb_staged_coord(kp, d, [&](int r) { return src[i * D + r]; }) : src[i * D + d];
    dst[(int64_t)d * np + i] = v;
}

__global__ void pad_cols_kernel(const double* __restrict__ src, int64_t n, int P, double* __restrict__ dst, int64_t np)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    int p = blockIdx.y;
    if (i >= np) return;
    dst[(int64_t)p * np + i] = (i < n) ? src[(int64_t)p * n + i] : 0.0;
}

__global__ void fill_kernel(double* __restrict__ p, int64_t n, double v)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// identity on the padding region rows/cols [n0, np)
__global__ void identity_pad_kernel(double* __restrict__ A, int64_t np, int64_t n0)
{
    int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    int64_t tot = np * np;
    for (; idx < tot; idx += (int64_t)gridDim.x * blockDim.x) {
        int64_t r = idx % np, c = idx / np;
        if (r >= n0 || c >= n0) A[idx] = (r == c) ? 1.0 : 0.0;
    }
}

__global__ void identity_blocks_kernel(double* __restrict__ invD, int b0, int b1)
{
    int b = b0 + blockIdx.x;
    if (b >= b1) return;
    double* p = invD + (int64_t)b * LB_TILE * LB_TILE;
    for (int idx = threadIdx.x; idx < LB_TILE * LB_TILE; idx += blockDim.x) p[idx] = ((idx & 127) == (idx >> 7)) ? 1.0 : 0.0;
}

// copy the N x N leading block of a column-major Np matrix, zeroing the strict upper part if asked
__global__ void extract_kernel(const double* __restrict__ A, int64_t np, int64_t n, double* __restrict__ dst, int lower_only)
{
    int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    int64_t tot = n * n;
    for (; idx < tot; idx += (int64_t)gridDim.x * blockDim.x) {
        int64_t r = idx % n, c = idx / n;
        double v = A[r + c * np];
        if (lower_only && r < c) v = 0.0;
        dst[idx] = v;
    }
}

// k(x_i, x_new) for i < n (no noise), zero beyond: kernel.hpp:81-84 with i != j
__global__ void krow_kernel(const double* __restrict__ Xs, int64_t np, int64_t n, int64_t inew, KernParams kp,
    double* __restrict__ out)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= np) return;
    double z = 0.0;
    for (int d = 0; d < kp.D; ++d) {
        double q = Xs[(int64_t)d * np + i] - Xs[(int64_t)d * np + inew];
        z = fma(q, q, z);
    }
    out[i] = (i < n) ? lb_kernel_from_z(kp.id, z, kp) : 0.0;
}

// finish the incremental row (gp.hpp:591-597): L[n, 0:n] = l^T ; L[n,n] = sqrt(k_nn - l.l)
__global__ void append_row_kernel(double* __restrict__ L, int64_t np, int64_t n, const double* __restrict__ lvec, double knn,
    int* __restrict__ info)
{
    __shared__ double red[8];
    double s = 0.0;
    for (int64_t j = threadIdx.x; j < n; j += blockDim.x) {
        double v = lvec[j];
        L[n + j * np] = v;
        s = fma(v, v, s);
    }
    s = lb_warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += red[w];
        double d = knn - t;
        if (!(d > 0.0)) atomicCAS(info, 0, (int)(n + 1));
        L[n + n * np] = sqrt(d);
    }
}

// callers synchronise the handle's stream first
void free_ws(QueryWs& w)
{
    void* all[] = {w.dQraw, w.dQs, w.dV, w.dMu, w.dS2, w.dAcq, w.dBlkVal, w.dBlkIdx, w.dBest, w.dBestIdx, w.dMean, w.dKt, w.dNorm2,
        w.dErr, w.dBias};
    for (void* p : all) lb_pool_free(p);
    w = QueryWs();
}

void free_model(lb_gp* h)
{
    void* all[] = {h->dX, h->dXs, h->dY, h->dL, h->dInvD, h->dAlpha, h->dLinv, h->dKinv, h->dFlags, h->dLinv32, h->dWork, h->dLinvW, h->dTrsvX,
        h->dLdig};
    h->dTrsvX = nullptr; h->trsvx_np = 0;
    h->dLdig = nullptr; h->ldig_np = 0; h->ldig_valid = false;
    for (void* p : all) lb_pool_free(p); // shared buffers (lb_clone) only lose this handle's reference
    h->dWork = nullptr; h->work_np = 0; h->dLinvW = nullptr; h->linvw_np = 0;
    h->dLinv32 = nullptr; h->linv32_valid = false; h->linv32_rows = 0;
    h->dX = h->dXs = h->dY = h->dL = h->dInvD = h->dAlpha = h->dLinv = h->dKinv = nullptr;
    h->dFlags = nullptr;
    h->Np = 0;
}

int alloc_model(lb_gp* h, int64_t Np, int D, int P)
{
    const int64_t T = Np / LB_TILE;
    LB_ALLOC(h, h->dX, sizeof(double) * D * Np);
    LB_ALLOC(h, h->dY, sizeof(double) * P * Np);
    LB_ALLOC(h, h->dFlags, sizeof(int) * (T + 8));
    h->Np = Np;
    return LB_OK; // Xs, L, invD, alpha: ensure_fit_buffers (a clone that refits never needs its source's copies)
}

// Private Xs / L / invD / alpha for a handle that is about to (re)factorise: allocated when missing, replaced without a
// copy when still shared with a clone (every byte is rewritten by the fit).
int ensure_fit_buffers(lb_gp* h)
{
    const int64_t Np = h->Np, T = Np / LB_TILE;
    int rc;
    bool fresh = false;
    if ((rc = make_unique(h, &h->dXs, sizeof(double) * (h->D + LB_MAX_LAMBDA) * Np, false))) return rc;
    if ((rc = make_unique(h, &h->dL, sizeof(double) * Np * Np, false))) return rc;
    if ((rc = make_unique(h, &h->dAlpha, sizeof(double) * h->P * Np, false))) return rc;
    if ((rc = make_unique(h, &h->dInvD, sizeof(double) * T * LB_TILE * LB_TILE, false, &fresh))) return rc;
    if (fresh) // the panel kernels only write the lower part of every block; consumers read whole blocks
        LB_CUDA(cudaMemsetAsync(h->dInvD, 0, sizeof(double) * T * LB_TILE * LB_TILE, h->stream));
    return LB_OK;
}

int check_info(lb_gp* h)
{
    int info[2] = {0, 0};
    LB_CUDA(cudaMemcpyAsync(info, h->dInfo, sizeof(info), cudaMemcpyDeviceToHost, h->stream));
    LB_CUDA(cudaStreamSynchronize(h->stream));
    if (info[1]) return LB_ERR_TIMEOUT;
    if (info[0] > 0) return info[0];
    return LB_OK;
}

int upload_kernel_scaled(lb_gp* h)
{
    if (h->N == 0 && h->Np == 0) return LB_OK;
    return lb_launch_scale_x(h);
}

} // namespace

int lb_ensure_scratch(lb_gp* h, size_t bytes)
{
    return ensure(h, &h->dScratch, &h->scratch_bytes, bytes);
}

extern "C" {
int lb_profile_enable(lb_gp* h, int on);

// Streams and events of destroyed handles are kept for the next lb_create on the same device: a likelihood
// evaluation clones and destroys one handle (kernel_lf_opt.hpp:79), and stream / event creation is not free either.
struct Shell { cudaStream_t own = nullptr, side = nullptr; cudaEvent_t ev[LB_NEV] = {}; };
static std::mutex g_shell_mu;
static std::vector<Shell> g_shells[64];

int lb_create(lb_gp** out, int device, int precision)
{
    if (!out) return LB_ERR_ARG;
    if (precision != LB_PREC_FP64 && precision != LB_PREC_TF32 && precision != LB_PREC_FP16 && precision != LB_PREC_FP16X3) return LB_ERR_UNSUPPORTED;
    int ndev = 0;
    LB_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev || device >= 64) return LB_ERR_ARG;
    lb_gp_full* h = new (std::nothrow) lb_gp_full();
    if (!h) return LB_ERR_ALLOC;
    h->device = device;
    DeviceGuard guard(h);
    if (!guard.ok) { delete h; return LB_ERR_CUDA; }
    h->precision = precision;
    Shell sh;
    bool cached = false;
    {
        std::lock_guard<std::mutex> lk(g_shell_mu);
        if (!g_shells[device].empty()) { sh = g_shells[device].back(); g_shells[device].pop_back(); cached = true; }
    }
    if (!cached) {
        if (cudaStreamCreateWithFlags(&sh.own, cudaStreamNonBlocking) != cudaSuccess) {
            delete h;
            return LB_ERR_CUDA;
        }
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        if (cudaStreamCreateWithPriority(&sh.side, cudaStreamNonBlocking, hi) != cudaSuccess) sh.side = nullptr;
        for (int i = 0; i < LB_NEV; ++i) cudaEventCreateWithFlags(&sh.ev[i], cudaEventDisableTiming);
    }
    h->ex.own = sh.own;
    h->stream = sh.own;
    h->own_stream = true;
    h->side = sh.side;
    for (int i = 0; i < LB_NEV; ++i) h->ev[i] = sh.ev[i];
    if (lb_dalloc(h, &h->dInfo, 4 * sizeof(int)) || lb_dalloc(h, &h->ex.dMisc, (LB_MAX_HPARAMS + 16) * sizeof(double))) {
        lb_destroy(h);
        return LB_ERR_ALLOC;
    }
    cudaMemsetAsync(h->dInfo, 0, 4 * sizeof(int), h->stream);
    h->kp.id = LB_K_SE_ARD;
    *out = h;
    return LB_OK;
}

int lb_destroy(lb_gp* hh)
{
    if (!hh) return LB_OK;
    lb_gp_full* h = full(hh);
    DeviceGuard guard(h);
    cudaStreamSynchronize(h->stream);
    if (h->ex.own && h->ex.own != h->stream) cudaStreamSynchronize(h->ex.own);
    if (h->side) cudaStreamSynchronize(h->side);
    lb_profile_enable(h, 0);
    free_model(h);
    free_ws(h->ex.ws);
    lb_pool_free(h->dInfo);
    lb_pool_free(h->dScratch);
    lb_pool_free(h->dLambda);
    lb_pool_free(h->ex.dMisc);
    if (h->ex.hPoint) cudaFreeHost(h->ex.hPoint);
    for (cudaStream_t* ps : {&h->aux, &h->aux2, &h->aux3})
        if (*ps) { cudaStreamSynchronize(*ps); cudaStreamDestroy(*ps); *ps = nullptr; }
    Shell sh;
    sh.own = h->ex.own; sh.side = h->side;
    for (int i = 0; i < LB_NEV; ++i) sh.ev[i] = h->ev[i];
    bool kept = false;
    if (sh.own && h->device >= 0 && h->device < 64) {
        std::lock_guard<std::mutex> lk(g_shell_mu);
        if (g_shells[h->device].size() < 64) { g_shells[h->device].push_back(sh); kept = true; }
    }
    if (!kept) {
        if (sh.own) cudaStreamDestroy(sh.own);
        if (sh.side) cudaStreamDestroy(sh.side);
        for (int i = 0; i < LB_NEV; ++i) if (sh.ev[i]) cudaEventDestroy(sh.ev[i]);
    }
    delete h;
    return LB_OK;
}

int lb_set_stream(lb_gp* h, void* s)
{
    if (!h) return LB_ERR_ARG;
    LB_DEVICE(h);
    lb_gp_full* f = full(h);
    LB_CUDA(cudaStreamSynchronize(f->stream));
    f->stream = s ? (cudaStream_t)s : f->ex.own;
    return LB_OK;
}

int lb_sync(lb_gp* h)
{
    if (!h) return LB_ERR_ARG;
    LB_DEVICE(h);
    LB_CUDA(cudaStreamSynchronize(h->stream));
    // device-side wait timeouts of the reduced-precision scoring path, for callers of the *_dev entry points (which
    // return before the kernels have run)
    lb_gp_full* f = full(h);
    if (f->ex.ws.dErr) {
        int herr = 0;
        LB_CUDA(cudaMemcpy(&herr, f->ex.ws.dErr, sizeof(int), cudaMemcpyDeviceToHost));
        if (herr) {
            LB_CUDA(cudaMemset(f->ex.ws.dErr, 0, sizeof(int)));
            return LB_ERR_TIMEOUT;
        }
    }
    return LB_OK;
}

long long lb_launch_count(const lb_gp* h) { return h ? h->launches : 0; }
int64_t lb_nb_samples(const lb_gp* h) { return h ? h->N : 0; }

static int set_data_common(lb_gp* h, int64_t N, int D, int P, const double* X, const double* Y, bool dev)
{
    if (!h || N < 0 || D < 1 || D > LB_MAX_D || P < 1) return LB_ERR_ARG;
    if (N > 0 && (!X || !Y)) return LB_ERR_ARG;
    LB_DEVICE(h);
    const int64_t Np = std::max<int64_t>(LB_TILE, (N + LB_TILE - 1) / LB_TILE * LB_TILE);
    if (Np != h->Np || D != h->D || P != h->P) {
        LB_CUDA(cudaStreamSynchronize(h->stream));
        free_model(h);
        int rc = alloc_model(h, Np, D, P);
        if (rc) return rc;
    }
    else { // same shape: rewrite in place unless a clone still reads the buffers
        int rc;
        if ((rc = make_unique(h, &h->dX, sizeof(double) * D * Np, false))) return rc;
        if ((rc = make_unique(h, &h->dY, sizeof(double) * P * Np, false))) return rc;
    }
    if (D != h->D) h->kp.klam = 0; // the Lambda matrix belongs to the previous input dimension
    h->N = N; h->D = D; h->P = P;
    h->kp.Draw = D;
    h->kp.D = D + h->kp.klam;
    h->fitted = false; h->linv_valid = false; h->linv_levels = 0; h->ldig_valid = false; h->kinv_valid = false; h->linv32_valid = false;
    const double* dXr = X;
    const double* dYr = Y;
    if (!dev && N > 0) {
        int rc = lb_ensure_scratch(h, sizeof(double) * (size_t)N * (D + P));
        if (rc) return rc;
        LB_CUDA(cudaMemcpyAsync(h->dScratch, X, sizeof(double) * N * D, cudaMemcpyHostToDevice, h->stream));
        LB_CUDA(cudaMemcpyAsync(h->dScratch + N * D, Y, sizeof(double) * N * P, cudaMemcpyHostToDevice, h->stream));
        dXr = h->dScratch;
        dYr = h->dScratch + N * D;
    }
    dim3 g1((unsigned)((Np + 255) / 256), (unsigned)D), g2((unsigned)((Np + 255) / 256), (unsigned)P);
    pack_soa_kernel<<<g1, 256, 0, h->stream>>>(dXr, N, D, h->dX, Np, h->kp, 0);
    pad_cols_kernel<<<g2, 256, 0, h->stream>>>(dYr, N, P, h->dY, Np);
    h->launches += 2;
    LB_CUDA(cudaGetLastError());
    return LB_OK;
}

// Samples only (multi-GPU Cholesky, potrf.cu lb_dchol_*): stages X without allocating the N x N factor storage of
// this handle; the handle can then only serve lb_set_kernel and the lb_dchol_* calls.
int lb_dchol_set_points(lb_gp* h, int64_t N, int D, const double* X)
{
    if (!h || N <= 0 || D < 1 || D > LB_MAX_D || !X) return LB_ERR_ARG;
    LB_DEVICE(h);
    LB_CUDA(cudaStreamSynchronize(h->stream));
    free_model(h);
    const int64_t Np = (N + LB_TILE - 1) / LB_TILE * LB_TILE;
    LB_ALLOC(h, h->dX, sizeof(double) * D * Np);
    LB_ALLOC(h, h->dXs, sizeof(double) * (D + LB_MAX_LAMBDA) * Np);
    h->Np = Np;
    if (D != h->D) h->kp.klam = 0;
    h->N = N; h->D = D; h->P = 0;
    h->kp.Draw = D;
    h->kp.D = D + h->kp.klam;
    h->fitted = false; h->linv_valid = false; h->linv_levels = 0; h->ldig_valid = false; h->kinv_valid = false; h->linv32_valid = false;
    int rc = lb_ensure_scratch(h, sizeof(double) * (size_t)N * D);
    if (rc) return rc;
    LB_CUDA(cudaMemcpyAsync(h->dScratch, X, sizeof(double) * N * D, cudaMemcpyHostToDevice, h->stream));
    dim3 g1((unsigned)((Np + 255) / 256), (unsigned)D);
    pack_soa_kernel<<<g1, 256, 0, h->stream>>>(h->dScratch, N, D, h->dX, Np, h->kp, 0);
    h->launches++;
    LB_CUDA(cudaStreamSynchronize(h->stream));
    LB_CUDA(cudaGetLastError());
    return LB_OK;
}

int lb_set_data(lb_gp* h, int64_t N, int D, int P, const double* X, const double* Y)
{
    return set_data_common(h, N, D, P, X, Y, false);
}
int lb_set_data_dev(lb_gp* h, int64_t N, int D, int P, const double* dX, const double* dY)
{
    return set_data_common(h, N, D, P, dX, dY, true);
}

int lb_set_kernel(lb_gp* h, int kernel_id, const double* p, int n_hparams, double noise)
{
    if (!h || !p) return LB_ERR_ARG;
    if (kernel_id < 0 || kernel_id > 3) return LB_ERR_UNSUPPORTED;
    if (h->D <= 0) return LB_ERR_STATE; // need the input dimension first (lb_set_data)
    int klam = 0;
    if (kernel_id == LB_K_SE_ARD) { // [log ell (D), A columns (D each, k of them), log sigma_f]  squared_exp_ard.hpp:91,96-105
        const int rest = n_hparams - 1 - h->D;
        if (rest < 0 || rest % h->D != 0) return LB_ERR_ARG;
        klam = rest / h->D;
        if (klam > LB_MAX_LAMBDA || h->D + klam > LB_MAX_D) return LB_ERR_UNSUPPORTED;
    }
    else if (n_hparams != 2)
        return LB_ERR_ARG;
    LB_DEVICE(h);
    bool lambda_same = true;
    const KernParams old = h->kp;
    const bool was_set = h->kernel_set;
    const int old_nh = h->n_hparams;
    KernParams& kp = h->kp;
    kp.id = kernel_id;
    kp.Draw = h->D;
    kp.klam = klam;
    kp.D = h->D + klam;
    kp.lambda = nullptr;
    kp.noise = noise;
    if (kernel_id == LB_K_SE_ARD) {
        for (int d = 0; d < h->D; ++d) kp.inv_ell[d] = 1.0 / std::exp(p[d]);
        kp.sf2 = std::exp(2.0 * p[n_hparams - 1]);
        kp.l = 1.0;
        if (klam > 0) { // _A(i, j) = p((j + 1) * D + i): already column-major
            if (!h->dLambda) LB_ALLOC(h, h->dLambda, sizeof(double) * LB_MAX_D * LB_MAX_LAMBDA);
            double* lh = full(h)->ex.lambda_host;
            lambda_same = (old.klam == klam) && std::memcmp(lh, p + h->D, sizeof(double) * h->D * klam) == 0;
            std::memcpy(lh, p + h->D, sizeof(double) * h->D * klam);
            LB_CUDA(cudaMemcpyAsync(h->dLambda, p + h->D, sizeof(double) * h->D * klam, cudaMemcpyHostToDevice, h->stream));
            LB_CUDA(cudaStreamSynchronize(h->stream));
            kp.lambda = h->dLambda;
        }
    }
    else { // matern_five_halves.hpp:97-102 and siblings
        kp.l = std::exp(p[0]);
        kp.sf2 = std::exp(2.0 * p[1]);
    }
    kp.c1 = kp.c2 = 0.0;
    if (kernel_id == LB_K_MATERN52) { kp.c1 = std::sqrt(5.0) / kp.l; kp.c2 = 5.0 / (3.0 * (kp.l * kp.l)); }
    else if (kernel_id == LB_K_MATERN32) kp.c1 = std::sqrt(3.0) / kp.l;
    else if (kernel_id == LB_K_EXP) kp.c1 = 1.0 / (kp.l * kp.l);
    h->n_hparams = n_hparams;
    h->kernel_set = true;
    // The same functor state again (add_sample pushes the kernel before every lb_append, gp.hpp:126-152 never touches
    // it): the factor stays valid.
    bool same = was_set && old_nh == n_hparams && klam == old.klam && lambda_same && old.id == kp.id && old.D == kp.D && old.Draw == kp.Draw
        && old.sf2 == kp.sf2 && old.l == kp.l && old.noise == kp.noise && old.c1 == kp.c1 && old.c2 == kp.c2;
    if (same && kernel_id == LB_K_SE_ARD)
        for (int d = 0; d < h->D; ++d) same = same && (old.inv_ell[d] == kp.inv_ell[d]);
    if (!same) { h->fitted = false; h->linv_valid = false; h->linv_levels = 0; h->ldig_valid = false; h->kinv_valid = false; h->linv32_valid = false; }
    return LB_OK;
}

int lb_fit(lb_gp* h)
{
    if (!h) return LB_ERR_ARG;
    if (!h->kernel_set || h->Np == 0 || !h->dX) return LB_ERR_STATE;
    LB_DEVICE(h);
    if (h->N == 0) return LB_ERR_STATE; // gp.hpp:90 assert(samples.size() != 0)
    int rc;
    if ((rc = ensure_fit_buffers(h))) return rc;
    if ((rc = lb_launch_scale_x(h))) return rc;
    if ((rc = lb_launch_kbuild(h, h->dL))) return rc;
    if ((rc = lb_launch_potrf(h))) return rc;
    h->fitted = true; h->linv_valid = false; h->linv_levels = 0; h->ldig_valid = false; h->kinv_valid = false; h->linv32_valid = false;
    if ((rc = lb_launch_solve_alpha(h))) return rc;
    return check_info(h);
}

int lb_fit_async(lb_gp* h) // same as lb_fit without the final host sync / info read (bench "value" leg)
{
    if (!h) return LB_ERR_ARG;
    if (!h->kernel_set || h->Np == 0 || h->N == 0 || !h->dX) return LB_ERR_STATE;
    LB_DEVICE(h);
    int rc;
    if ((rc = ensure_fit_buffers(h))) return rc;
    if ((rc = lb_launch_scale_x(h))) return rc;
    if ((rc = lb_launch_kbuild(h, h->dL))) return rc;
    if ((rc = lb_launch_potrf(h))) return rc;
    h->fitted = true; h->linv_valid = false; h->linv_levels = 0; h->ldig_valid = false; h->kinv_valid = false; h->linv32_valid = false;
    return lb_launch_solve_alpha(h);
}

int lb_check_info(lb_gp* h)
{
    if (!h) return LB_ERR_ARG;
    LB_DEVICE(h);
    return check_info(h);
}
int lb_debug_potf2(lb_gp* h, int k, long long* out, int n)
{
    if (!h) return LB_ERR_ARG;
    LB_DEVICE(h);
    return lb_debug_potf2_clocks(h, k, out, n);
}
// testing hook: how many times lb_append took the incremental path on this handle
long long lb_debug_append_count(const lb_gp* h) { return h ? full(h)->ex.n_append : 0; }
// testing hook: force the multi-launch (unfused) query path
int lb_debug_force_unfused_query(lb_gp* h, int on) { if (!h) return LB_ERR_ARG; h->force_unfused = on != 0; return LB_OK; }

// stage timers for bench.py: run only one stage (inputs must already be in place)
int lb_stage_kbuild(lb_gp* h)
{
    if (!h || !h->kernel_set || h->N == 0) return LB_ERR_STATE;
    LB_DEVICE(h);
    int rc;
    if ((rc = ensure_fit_buffers(h))) return rc;
    if ((rc = lb_launch_scale_x(h))) return rc;
    h->fitted = false;
    return lb_launch_kbuild(h, h->dL);
}
int lb_stage_potrf(lb_gp* h)
{
    if (!h || h->N == 0 || !h->dL) return LB_ERR_STATE;
    LB_DEVICE(h);
    int rc = lb_launch_potrf(h);
    if (!rc) h->fitted = true;
    return rc;
}
int lb_stage_alpha(lb_gp* h)
{
    if (!h || !h->fitted) return LB_ERR_STATE;
    LB_DEVICE(h);
    return lb_launch_solve_alpha(h);
}

// GP::load(archive, recompute = false) (gp.hpp:505-509): take a stored factor and alpha instead of refactorising.
// Data and kernel must already be set (lb_set_data / lb_set_kernel); the diagonal-block inverses are rebuilt.
int lb_load_factor(lb_gp* h, const double* L_colmajor, const double* alpha_colmajor)
{
    if (!h || !L_colmajor || !alpha_colmajor) return LB_ERR_ARG;
    if (!h->kernel_set || h->N == 0 || h->Np == 0) return LB_ERR_STATE;
    LB_DEVICE(h);
    const int64_t N = h->N, Np = h->Np;
    const int T = (int)(Np / LB_TILE);
    int rc;
    if ((rc = ensure_fit_buffers(h))) return rc;
    if ((rc = lb_launch_scale_x(h))) return rc;
    LB_CUDA(cudaMemsetAsync(h->dL, 0, sizeof(double) * Np * Np, h->stream));
    LB_CUDA(cudaMemcpy2DAsync(h->dL, Np * 8, L_colmajor, N * 8, N * 8, N, cudaMemcpyHostToDevice, h->stream));
    identity_pad_kernel<<<1024, 256, 0, h->stream>>>(h->dL, Np, N);
    LB_CUDA(cudaMemsetAsync(h->dAlpha, 0, sizeof(double) * Np * h->P, h->stream));
    LB_CUDA(cudaMemcpy2DAsync(h->dAlpha, Np * 8, alpha_colmajor, N * 8, N * 8, h->P, cudaMemcpyHostToDevice, h->stream));
    LB_CUDA(cudaMemsetAsync(h->dInfo, 0, 2 * sizeof(int), h->stream));
    h->launches++;
    for (int k = 0; k < T; ++k)
        if ((rc = lb_launch_potf2_block(h, k, 0))) return rc;
    h->fitted = true; h->linv_valid = false; h->linv_levels = 0; h->ldig_valid = false; h->kinv_valid = false; h->linv32_valid = false;
    return check_info(h);
}

int lb_refit_alpha(lb_gp* h, const double* Y)
{
    if (!h || !Y) return LB_ERR_ARG;
    if (!h->fitted) return LB_ERR_STATE;
    LB_DEVICE(h);
    int rc = lb_ensure_scratch(h, sizeof(double) * (size_t)h->N * h->P);
    if (rc) return rc;
    if ((rc = make_unique(h, &h->dY, sizeof(double) * h->P * h->Np, false))) return rc;
    if ((rc = make_unique(h, &h->dAlpha, sizeof(double) * h->P * h->Np, false))) return rc;
    LB_CUDA(cudaMemcpyAsync(h->dScratch, Y, sizeof(double) * h->N * h->P, cudaMemcpyHostToDevice, h->stream));
    dim3 g2((unsigned)((h->Np + 255) / 256), (unsigned)h->P);
    pad_cols_kernel<<<g2, 256, 0, h->stream>>>(h->dScratch, h->N, h->P, h->dY, h->Np);
    h->launches++;
    if ((rc = lb_launch_solve_alpha(h))) return rc;
    return check_info(h);
}

int lb_append(lb_gp* h, const double* x, const double* Yall)
{
    if (!h || !x || !Yall) return LB_ERR_ARG;
    if (!h->kernel_set) return LB_ERR_STATE;
    LB_DEVICE(h);
    if (h->N == 0 || !h->fitted) return LB_ERR_STATE; // first sample goes through lb_set_data + lb_fit
    const int64_t n = h->N;
    const int D = h->D, P = h->P;
    if (n + 1 > h->Np) { // grow by one tile, keep the factor
        const int64_t oldNp = h->Np, newNp = oldNp + LB_TILE;
        const int64_t oldT = oldNp / LB_TILE, newT = newNp / LB_TILE;
        double *nX, *nXs, *nY, *nA, *nL, *nI; int* nF;
        LB_CUDA(cudaStreamSynchronize(h->stream));
        LB_ALLOC(h, nX, sizeof(double) * D * newNp);
        LB_ALLOC(h, nXs, sizeof(double) * (D + LB_MAX_LAMBDA) * newNp);
        LB_ALLOC(h, nY, sizeof(double) * P * newNp);
        LB_ALLOC(h, nA, sizeof(double) * P * newNp);
        LB_ALLOC(h, nL, sizeof(double) * newNp * newNp);
        LB_ALLOC(h, nI, sizeof(double) * newT * LB_TILE * LB_TILE);
        LB_ALLOC(h, nF, sizeof(int) * (newT + 8));
        LB_CUDA(cudaMemsetAsync(nX, 0, sizeof(double) * D * newNp, h->stream));
        LB_CUDA(cudaMemsetAsync(nY, 0, sizeof(double) * P * newNp, h->stream));
        LB_CUDA(cudaMemcpy2DAsync(nX, newNp * 8, h->dX, oldNp * 8, oldNp * 8, D, cudaMemcpyDeviceToDevice, h->stream));
        LB_CUDA(cudaMemcpy2DAsync(nL, newNp * 8, h->dL, oldNp * 8, oldNp * 8, oldNp, cudaMemcpyDeviceToDevice, h->stream));
        LB_CUDA(cudaMemcpyAsync(nI, h->dInvD, sizeof(double) * oldT * LB_TILE * LB_TILE, cudaMemcpyDeviceToDevice, h->stream));
        identity_pad_kernel<<<1024, 256, 0, h->stream>>>(nL, newNp, oldNp);
        identity_blocks_kernel<<<(unsigned)(newT - oldT), 256, 0, h->stream>>>(nI, (int)oldT, (int)newT);
        h->launches += 2;
        LB_CUDA(cudaStreamSynchronize(h->stream));
        lb_pool_free(h->dX); lb_pool_free(h->dXs); lb_pool_free(h->dY); lb_pool_free(h->dAlpha); lb_pool_free(h->dL); lb_pool_free(h->dInvD);
        lb_pool_free(h->dFlags); lb_pool_free(h->dLinv); lb_pool_free(h->dKinv);
        h->dX = nX; h->dXs = nXs; h->dY = nY; h->dAlpha = nA; h->dL = nL; h->dInvD = nI; h->dFlags = nF;
        h->dLinv = h->dKinv = nullptr;
        h->Np = newNp;
    }
    const int64_t Np = h->Np;
    int rc = lb_ensure_scratch(h, sizeof(double) * (size_t)((n + 1) * P + D + Np));
    if (rc) return rc;
    { // copy-on-write: a clone may still read these (the row update keeps the rest of X, L, invD)
        const int64_t T = Np / LB_TILE;
        if ((rc = make_unique(h, &h->dX, sizeof(double) * D * Np, true))) return rc;
        if ((rc = make_unique(h, &h->dL, sizeof(double) * Np * Np, true))) return rc;
        if ((rc = make_unique(h, &h->dInvD, sizeof(double) * T * LB_TILE * LB_TILE, true))) return rc;
        if ((rc = make_unique(h, &h->dY, sizeof(double) * P * Np, false))) return rc;
        if ((rc = make_unique(h, &h->dXs, sizeof(double) * (D + LB_MAX_LAMBDA) * Np, false))) return rc;
        if ((rc = make_unique(h, &h->dAlpha, sizeof(double) * P * Np, false))) return rc;
    }
    full(h)->ex.n_append++;
    double* dYs = h->dScratch;
    double* dx = dYs + (n + 1) * P;
    double* dk = dx + D;
    LB_CUDA(cudaMemcpyAsync(dYs, Yall, sizeof(double) * (n + 1) * P, cudaMemcpyHostToDevice, h->stream));
    LB_CUDA(cudaMemcpyAsync(dx, x, sizeof(double) * D, cudaMemcpyHostToDevice, h->stream));
    // X[:, n] = x  (strided D writes)
    LB_CUDA(cudaMemcpy2DAsync(h->dX + n, Np * 8, dx, 8, 8, D, cudaMemcpyDeviceToDevice, h->stream));
    h->N = n + 1;
    dim3 g2((unsigned)((Np + 255) / 256), (unsigned)P);
    pad_cols_kernel<<<g2, 256, 0, h->stream>>>(dYs, n + 1, P, h->dY, Np);
    h->launches++;
    if ((rc = lb_launch_scale_x(h))) return rc;
    // new kernel row (gp.hpp:583-586), forward solve against the existing factor (gp.hpp:591-594)
    krow_kernel<<<(unsigned)((Np + 255) / 256), 256, 0, h->stream>>>(h->dXs, Np, n, n, h->kp, dk);
    h->launches++;
    if ((rc = lb_launch_trsv(h, dk, 1, true))) return rc;
    const double knn = h->kp.sf2 + h->kp.noise + 1e-8; // kernel(x,x) with i == j, kernel.hpp:83
    append_row_kernel<<<1, 256, 0, h->stream>>>(h->dL, Np, n, dk, knn, h->dInfo);
    h->launches++;
    if ((rc = lb_launch_potf2_block(h, (int)(n / LB_TILE), 0))) return rc;
    h->linv_valid = false; h->linv_levels = 0; h->ldig_valid = false; h->kinv_valid = false; h->linv32_valid = false;
    if ((rc = lb_launch_solve_alpha(h))) return rc;
    return check_info(h);
}

// Batches of at least this many candidates take the panel path (LB_QUERY_PANEL_MIN overrides).  The slab kernel keeps the
// one-point / small-batch latency, but its time does not shrink with the batch: every CTA streams all of L through L2 whatever
// its slab width (N = 16384: ~88 ms for ANY batch of <= 10^4 candidates; measured on 8 GPUs, 1250 candidates per rank), while
// the panel path scales with the number of 128-candidate column tiles.
static int64_t g_query_panel_min = -1;
static int64_t query_panel_min()
{
    if (g_query_panel_min < 0) {
        const char* e = getenv("LB_QUERY_PANEL_MIN");
        int64_t v = e ? (int64_t)atoll(e) : 256;
        g_query_panel_min = v < 1 ? 1 : v;
    }
    return g_query_panel_min;
}
// testing hook: batch size from which lb_query / lb_acq_argmax take the panel path (<= 0 restores the default)
extern "C" int lb_debug_set_query_panel_min(long long m)
{
    g_query_panel_min = m > 0 ? (int64_t)m : -1;
    return LB_OK;
}

static int query_common(const lb_gp* hc, int64_t M, const double* Xq, bool xq_dev, double* mu_out, double* s2_out,
    bool out_dev, int acq_id, const double* acq_params, const double* mean_at_q, double mean_const, double* acq_out,
    double* best_val, int64_t* best_idx, bool with_acq)
{
    if (!hc || M < 0) return LB_ERR_ARG;
    if (M == 0) return LB_OK;
    if (!Xq) return LB_ERR_ARG;
    lb_gp_full* h = full(hc);
    if (h->D <= 0 || !h->kernel_set) return LB_ERR_STATE;
    LB_DEVICE(h);
    std::lock_guard<std::mutex> lock(h->ex.qmutex);
    QueryWs& w = h->ex.ws;
    cudaStream_t st = h->stream;
    const int D = h->D, De = h->kp.D, P = h->P > 0 ? h->P : 1; // raw / staged input dimension
    const int64_t Mp = (M + LB_TILE - 1) / LB_TILE * LB_TILE;
    int rc;
    if ((rc = ensure(h, &w.dMu, &w.mu_bytes, sizeof(double) * M * P))) return rc;
    if ((rc = ensure(h, &w.dS2, &w.s2_bytes, sizeof(double) * M))) return rc;
    const bool prior = (h->N == 0 || !h->fitted);
    if (prior && h->N != 0) return LB_ERR_STATE;
    if (M == 1 && !prior && !xq_dev && !out_dev && !with_acq && h->precision == LB_PREC_FP64 && lb_query_fused_supported(h) && !h->force_unfused) {
        // one launch, one synchronisation (query.cu: query_point_kernel)
        Extra& ex = h->ex;
        if (ex.point_cap < P + 1) {
            if (ex.hPoint) cudaFreeHost(ex.hPoint);
            ex.hPoint = ex.dPoint = nullptr;
            LB_CUDA(cudaHostAlloc((void**)&ex.hPoint, sizeof(double) * (P + 1 + 7), cudaHostAllocMapped));
            LB_CUDA(cudaHostGetDevicePointer((void**)&ex.dPoint, ex.hPoint, 0));
            ex.point_cap = P + 1 + 7;
        }
        if ((rc = ensure(h, &w.dQs, &w.qs_bytes, sizeof(double) * De * LB_TILE))) return rc;
        if ((rc = ensure(h, &w.dV, &w.v_bytes, sizeof(double) * lb_query_fused_scratch_doubles(h, 1)))) return rc;
        if ((rc = lb_launch_query_point(h, st, Xq, w.dQs, w.dV, ex.dPoint, &h->launches))) return rc;
        LB_CUDA(cudaStreamSynchronize(st));
        if (mu_out) std::memcpy(mu_out, ex.hPoint, sizeof(double) * P);
        if (s2_out) *s2_out = ex.hPoint[P];
        return LB_OK;
    }
    if (prior) { // gp.hpp:161-163: mu = mean(v) (added by the caller), sigma2 = k(v,v) + noise
        LB_CUDA(cudaMemsetAsync(w.dMu, 0, sizeof(double) * M * P, st));
        fill_kernel<<<(unsigned)((M + 255) / 256), 256, 0, st>>>(w.dS2, M, h->kp.sf2 + h->kp.noise);
        h->launches++;
    }
    else {
        const double* dQraw = Xq;
        if (!xq_dev) {
            if ((rc = ensure(h, &w.dQraw, &w.qraw_bytes, sizeof(double) * M * D))) return rc;
            LB_CUDA(cudaMemcpyAsync(w.dQraw, Xq, sizeof(double) * M * D, cudaMemcpyHostToDevice, st));
            dQraw = w.dQraw;
        }
        if (h->precision == LB_PREC_TF32 || h->precision == LB_PREC_FP16 || h->precision == LB_PREC_FP16X3) {
            // reduced-precision variance on tcgen05 (tf32_query.cu); mu is accumulated in fp64 from the fp64 kernel values
            if ((rc = lb_tf32_prepare(h))) return rc;
            // Candidate chunks of k x (SMs / 2 CTA pairs x 256 candidates): whole waves of the persistent tcgen05 GEMM (a 65536
            // chunk = 3.46 waves cost 15 %); K*^T chunk <= 4 GiB.
            int sms = 148;
            LB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device));
            const int64_t CH = 2 * LB_TILE, wave = (int64_t)(sms / 2) * CH;
            const int64_t cap = std::max<int64_t>(CH, ((int64_t)4 << 30) / (4 * h->Np) / CH * CH);
            int64_t Mc = (cap >= wave) ? cap / wave * wave : cap;
            Mc = std::min((M + CH - 1) / CH * CH, Mc);
            if ((rc = ensure(h, &w.dQs, &w.qs_bytes, sizeof(double) * De * Mc))) return rc;
            if ((rc = ensure(h, &w.dKt, &w.kt_bytes, sizeof(float) * (size_t)Mc * h->Np))) return rc;
            if ((rc = ensure(h, &w.dNorm2, &w.norm2_bytes, sizeof(float) * (size_t)Mc * 4))) return rc; // up to 4 cluster partials (split mode: Mc doubles)
            if ((rc = ensure(h, &w.dV, &w.v_bytes, sizeof(double) * (size_t)(P + 1) * (h->Np / LB_TILE) * Mc))) return rc; // mean (+ bias) partials per training tile
            if ((rc = ensure(h, &w.dBias, &w.bias_bytes, sizeof(double) * Mc))) return rc;
            double* dBiasUse = (h->precision == LB_PREC_FP16X3) ? nullptr : w.dBias; // 22-bit operands: no rounding-bias term
            if (!w.dErr) LB_ALLOC(h, w.dErr, sizeof(int));
            LB_CUDA(cudaMemsetAsync(w.dErr, 0, sizeof(int), st));
            for (int64_t m0 = 0; m0 < M; m0 += Mc) {
                const int64_t mc = std::min(Mc, M - m0);
                const int64_t mcp = (mc + CH - 1) / CH * CH;
                dim3 g1((unsigned)((mcp + 255) / 256), (unsigned)De);
                pack_soa_kernel<<<g1, 256, 0, st>>>(dQraw + m0 * D, mc, D, w.dQs, mcp, h->kp, 1);
                h->launches++;
                if ((rc = lb_launch_kstar_tf32(h, st, mc, w.dQs, mcp, w.dKt, w.dV, w.dMu + m0 * P, dBiasUse, &h->launches))) return rc;
                if ((rc = lb_launch_sigma_tf32(h, st, mc, mcp, w.dKt, w.dNorm2, w.dErr, dBiasUse, w.dS2 + m0, &h->launches))) return rc;
            }
            if (!out_dev) {
                int herr = 0;
                LB_CUDA(cudaMemcpyAsync(&herr, w.dErr, sizeof(int), cudaMemcpyDeviceToHost, st));
                LB_CUDA(cudaStreamSynchronize(st));
                if (herr) return LB_ERR_TIMEOUT;
            }
        }
        else if (M >= query_panel_min() && !h->force_unfused) {
            // large batches: blocked solve over 2048-row super-blocks on the GEMM core (query.cu, namespace panel);
            // candidate chunks bounded so that V (Np x Mc) stays <= ~6 GiB
            const int64_t maxcols = std::max<int64_t>(LB_TILE, ((int64_t)6 << 30) / (8 * h->Np) / LB_TILE * LB_TILE);
            const int64_t Mc = std::min(Mp, maxcols);
            if ((rc = ensure(h, &w.dQs, &w.qs_bytes, sizeof(double) * De * Mc))) return rc;
            if ((rc = ensure(h, &w.dV, &w.v_bytes, sizeof(double) * lb_query_panel_scratch_doubles(h, Mc)))) return rc;
            const bool i8 = lb_query_int8_mode() != 0; // the int8 update's mbarrier waits are bounded and raise w.dErr
            if (i8) {
                if (!w.dErr) LB_ALLOC(h, w.dErr, sizeof(int));
                LB_CUDA(cudaMemsetAsync(w.dErr, 0, sizeof(int), st));
            }
            for (int64_t m0 = 0; m0 < M; m0 += Mc) {
                const int64_t mc = std::min(Mc, M - m0);
                const int64_t mcp = (mc + LB_TILE - 1) / LB_TILE * LB_TILE;
                dim3 g1((unsigned)((mcp + 255) / 256), (unsigned)De);
                pack_soa_kernel<<<g1, 256, 0, st>>>(dQraw + m0 * D, mc, D, w.dQs, mcp, h->kp, 1);
                h->launches++;
                if ((rc = lb_launch_query_panel(h, st, mc, w.dQs, mcp, w.dV, w.dMu + m0 * P, w.dS2 + m0, w.dErr, &h->launches))) return rc;
            }
            if (i8 && !out_dev) {
                int herr = 0;
                LB_CUDA(cudaMemcpyAsync(&herr, w.dErr, sizeof(int), cudaMemcpyDeviceToHost, st));
                LB_CUDA(cudaStreamSynchronize(st));
                if (herr) return LB_ERR_TIMEOUT;
            }
        }
        else if (lb_query_fused_supported(h) && !h->force_unfused) {
            // fused persistent path: one CTA per candidate slab, private V scratch per CTA
            int sms = 0;
            LB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device));
            const int64_t ntiles = (M + 7) / 8;
            const int grid = (int)std::min<int64_t>(sms, ntiles);
            if ((rc = ensure(h, &w.dQs, &w.qs_bytes, sizeof(double) * De * Mp))) return rc;
            if ((rc = ensure(h, &w.dV, &w.v_bytes, sizeof(double) * lb_query_fused_scratch_doubles(h, grid)))) return rc;
            dim3 g1((unsigned)((Mp + 255) / 256), (unsigned)De);
            pack_soa_kernel<<<g1, 256, 0, st>>>(dQraw, M, D, w.dQs, Mp, h->kp, 1);
            h->launches++;
            if ((rc = lb_launch_query_fused(h, st, M, w.dQs, Mp, w.dV, grid, w.dMu, w.dS2, &h->launches))) return rc;
        }
        else {
        // candidate chunks bounded so that V (Np x Mc) stays <= ~4 GiB
        int64_t Mc = Mp;
        const int64_t maxcols = std::max<int64_t>(LB_TILE, ((int64_t)4 << 30) / (8 * h->Np) / LB_TILE * LB_TILE);
        if (Mc > maxcols) Mc = maxcols;
        if ((rc = ensure(h, &w.dQs, &w.qs_bytes, sizeof(double) * De * Mc))) return rc;
        if ((rc = ensure(h, &w.dV, &w.v_bytes, sizeof(double) * h->Np * Mc))) return rc;
        for (int64_t m0 = 0; m0 < M; m0 += Mc) {
            const int64_t mc = std::min(Mc, M - m0);
            const int64_t mcp = (mc + LB_TILE - 1) / LB_TILE * LB_TILE;
            dim3 g1((unsigned)((mcp + 255) / 256), (unsigned)De);
            pack_soa_kernel<<<g1, 256, 0, st>>>(dQraw + m0 * D, mc, D, w.dQs, mcp, h->kp, 1);
            h->launches++;
            if ((rc = lb_launch_query(h, st, mc, w.dQs, mcp, w.dV, w.dMu + m0 * P, w.dS2 + m0, &h->launches))) return rc;
        }
        }
    }
    if (with_acq) {
        const int nblk = (int)((M + 255) / 256);
        if ((size_t)nblk > w.blk_cap) {
            lb_dfree_sync(h, w.dBlkVal); lb_dfree_sync(h, w.dBlkIdx);
            w.dBlkVal = nullptr; w.dBlkIdx = nullptr; w.blk_cap = 0;
            LB_ALLOC(h, w.dBlkVal, sizeof(double) * nblk);
            LB_ALLOC(h, w.dBlkIdx, sizeof(long long) * nblk);
            w.blk_cap = nblk;
        }
        if (!w.dBest) {
            LB_ALLOC(h, w.dBest, sizeof(double));
            LB_ALLOC(h, w.dBestIdx, sizeof(long long));
        }
        const double* dMean = nullptr;
        if (mean_at_q) {
            if (out_dev) dMean = mean_at_q;
            else {
                if ((rc = ensure(h, &w.dMean, &w.mean_bytes, sizeof(double) * M))) return rc;
                LB_CUDA(cudaMemcpyAsync(w.dMean, mean_at_q, sizeof(double) * M, cudaMemcpyHostToDevice, st));
                dMean = w.dMean;
            }
        }
        double* dAcq = nullptr;
        if (acq_out) {
            if (out_dev) dAcq = acq_out;
            else {
                if ((rc = ensure(h, &w.dAcq, &w.acq_bytes, sizeof(double) * M))) return rc;
                dAcq = w.dAcq;
            }
        }
        double* dBV = out_dev ? best_val : w.dBest;
        long long* dBI = out_dev ? (long long*)best_idx : w.dBestIdx;
        const double p0 = acq_params ? acq_params[0] : 0.0;
        const double p1 = (acq_params && acq_id == LB_ACQ_EI) ? acq_params[1] : 0.0;
        if ((rc = lb_launch_acq_full(st, acq_id, p0, p1, M, w.dMu, P, dMean, mean_const, w.dS2, dAcq, w.dBlkVal, w.dBlkIdx,
                 dBV, dBI, &h->launches)))
            return rc;
        if (!out_dev) {
            if (acq_out) LB_CUDA(cudaMemcpyAsync(acq_out, w.dAcq, sizeof(double) * M, cudaMemcpyDeviceToHost, st));
            long long bi = 0;
            LB_CUDA(cudaMemcpyAsync(best_val, w.dBest, sizeof(double), cudaMemcpyDeviceToHost, st));
            LB_CUDA(cudaMemcpyAsync(&bi, w.dBestIdx, sizeof(long long), cudaMemcpyDeviceToHost, st));
            LB_CUDA(cudaStreamSynchronize(st));
            *best_idx = (int64_t)bi;
        }
    }
    if (mu_out) {
        LB_CUDA(cudaMemcpyAsync(mu_out, w.dMu, sizeof(double) * M * P, out_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
    }
    if (s2_out) {
        LB_CUDA(cudaMemcpyAsync(s2_out, w.dS2, sizeof(double) * M, out_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
    }
    if (!out_dev) LB_CUDA(cudaStreamSynchronize(st));
    LB_CUDA(cudaGetLastError());
    return LB_OK;
}

int lb_query(const lb_gp* h, int64_t M, const double* Xq, double* mu, double* s2)
{
    return query_common(h, M, Xq, false, mu, s2, false, 0, nullptr, nullptr, 0.0, nullptr, nullptr, nullptr, false);
}
int lb_query_dev(const lb_gp* h, int64_t M, const double* dXq, double* dMu, double* dS2)
{
    return query_common(h, M, dXq, true, dMu, dS2, true, 0, nullptr, nullptr, 0.0, nullptr, nullptr, nullptr, false);
}

int lb_acq_argmax(const lb_gp* h, int acq_id, const double* acq_params, int64_t M, const double* Xq, const double* mean_at_q,
    double mean_const, double* acq_out, double* best_val, int64_t* best_idx)
{
    if (!best_val || !best_idx || !acq_params || M <= 0) return LB_ERR_ARG;
    if (acq_id != LB_ACQ_UCB && acq_id != LB_ACQ_EI) return LB_ERR_UNSUPPORTED;
    return query_common(h, M, Xq, false, nullptr, nullptr, false, acq_id, acq_params, mean_at_q, mean_const, acq_out, best_val,
        best_idx, true);
}
int lb_acq_argmax_dev(const lb_gp* h, int acq_id, const double* acq_params, int64_t M, const double* dXq,
    const double* dMean_at_q, double mean_const, double* dAcq_out, double* dBest_val, int64_t* dBest_idx)
{
    if (!dBest_val || !dBest_idx || !acq_params || M <= 0) return LB_ERR_ARG;
    if (acq_id != LB_ACQ_UCB && acq_id != LB_ACQ_EI) return LB_ERR_UNSUPPORTED;
    return query_common(h, M, dXq, true, nullptr, nullptr, true, acq_id, acq_params, dMean_at_q, mean_const, dAcq_out,
        dBest_val, dBest_idx, true);
}

int lb_log_lik(lb_gp* hh, double* out)
{
    if (!hh || !out) return LB_ERR_ARG;
    if (!hh->fitted) return LB_ERR_STATE;
    LB_DEVICE(hh);
    lb_gp_full* h = full(hh);
    int rc = lb_launch_loglik(h, h->ex.dMisc);
    if (rc) return rc;
    double v[3];
    LB_CUDA(cudaMemcpyAsync(v, h->ex.dMisc, sizeof(v), cudaMemcpyDeviceToHost, h->stream));
    LB_CUDA(cudaStreamSynchronize(h->stream));
    *out = v[2];
    return LB_OK;
}

int lb_compute_inv_kernel(lb_gp* h)
{
    if (!h) return LB_ERR_ARG;
    if (!h->fitted) return LB_ERR_STATE;
    if (h->kinv_valid) return LB_OK;
    LB_DEVICE(h);
    return lb_launch_kinv(h);
}

int lb_kernel_grad_log_lik(lb_gp* hh, int optimize_noise, double* grad)
{
    if (!hh || !grad) return LB_ERR_ARG;
    if (!hh->fitted) return LB_ERR_STATE;
    LB_DEVICE(hh);
    lb_gp_full* h = full(hh);
    int rc;
    if (!h->kinv_valid && (rc = lb_launch_kinv(h))) return rc;
    const int nh = h->n_hparams + (optimize_noise ? 1 : 0);
    if (nh > LB_MAX_HPARAMS) return LB_ERR_ARG;
    if ((rc = lb_launch_grad(h, optimize_noise, h->ex.dMisc + 8))) return rc;
    LB_CUDA(cudaMemcpyAsync(grad, h->ex.dMisc + 8, sizeof(double) * nh, cudaMemcpyDeviceToHost, h->stream));
    LB_CUDA(cudaStreamSynchronize(h->stream));
    return LB_OK;
}

int lb_log_loo_cv(lb_gp* hh, double* out)
{
    if (!hh || !out) return LB_ERR_ARG;
    if (!hh->fitted) return LB_ERR_STATE;
    LB_DEVICE(hh);
    lb_gp_full* h = full(hh);
    int rc = lb_launch_loo_value(h, h->ex.dMisc + 4);
    if (rc) return rc;
    LB_CUDA(cudaMemcpyAsync(out, h->ex.dMisc + 4, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    LB_CUDA(cudaStreamSynchronize(h->stream));
    return LB_OK;
}

int lb_kernel_grad_log_loo_cv(lb_gp* hh, int optimize_noise, double* grad)
{
    if (!hh || !grad) return LB_ERR_ARG;
    if (!hh->fitted) return LB_ERR_STATE;
    LB_DEVICE(hh);
    lb_gp_full* h = full(hh);
    const int nh = h->n_hparams + (optimize_noise ? 1 : 0);
    if (nh > LB_MAX_HPARAMS) return LB_ERR_ARG;
    int rc = lb_launch_loo_grad(h, optimize_noise, h->ex.dMisc + 8);
    if (rc) return rc;
    LB_CUDA(cudaMemcpyAsync(grad, h->ex.dMisc + 8, sizeof(double) * nh, cudaMemcpyDeviceToHost, h->stream));
    LB_CUDA(cudaStreamSynchronize(h->stream));
    return LB_OK;
}

int lb_kinv_obs_mean(lb_gp* h, double* out)
{
    if (!h || !out) return LB_ERR_ARG;
    if (!h->fitted) return LB_ERR_STATE;
    LB_DEVICE(h);
    double* dOut = nullptr;
    LB_ALLOC(h, dOut, sizeof(double) * h->N * h->P);
    int rc = lb_launch_kinv_obs(h, dOut);
    if (!rc) {
        if (cudaMemcpyAsync(out, dOut, sizeof(double) * h->N * h->P, cudaMemcpyDeviceToHost, h->stream) != cudaSuccess
            || cudaStreamSynchronize(h->stream) != cudaSuccess)
            rc = LB_ERR_CUDA;
    }
    lb_dfree_sync(h, dOut);
    return rc;
}

int lb_get(lb_gp* h, int what, double* dst)
{
    if (!h || !dst) return LB_ERR_ARG;
    if (h->N == 0) return LB_ERR_STATE;
    LB_DEVICE(h);
    const int64_t N = h->N, Np = h->Np;
    int rc;
    if (what == LB_GET_ALPHA) {
        if (!h->fitted) return LB_ERR_STATE;
        LB_CUDA(cudaMemcpy2DAsync(dst, N * 8, h->dAlpha, Np * 8, N * 8, h->P, cudaMemcpyDeviceToHost, h->stream));
        LB_CUDA(cudaStreamSynchronize(h->stream));
        return LB_OK;
    }
    if ((rc = lb_ensure_scratch(h, sizeof(double) * (size_t)(Np * Np + N * N)))) return rc;
    double* dTmp = h->dScratch;
    double* dOut = h->dScratch + Np * Np;
    const double* src = nullptr;
    int lower = 0;
    if (what == LB_GET_K) {
        if (!h->kernel_set) return LB_ERR_STATE;
        if ((rc = make_unique(h, &h->dXs, sizeof(double) * (h->D + LB_MAX_LAMBDA) * Np, false))) return rc;
        if ((rc = lb_launch_scale_x(h))) return rc;
        if ((rc = lb_launch_kbuild(h, dTmp))) return rc;
        src = dTmp;
    }
    else if (what == LB_GET_L) {
        if (!h->fitted) return LB_ERR_STATE;
        src = h->dL;
        lower = 1;
    }
    else if (what == LB_GET_KINV) {
        if (!h->fitted) return LB_ERR_STATE;
        if (!h->kinv_valid && (rc = lb_launch_kinv(h))) return rc;
        if (!h->kinv_sym) {
            if ((rc = lb_launch_symmetrize(h, h->dKinv))) return rc;
            h->kinv_sym = true;
        }
        src = h->dKinv;
    }
    else
        return LB_ERR_ARG;
    extract_kernel<<<1024, 256, 0, h->stream>>>(src, Np, N, dOut, lower);
    h->launches++;
    LB_CUDA(cudaMemcpyAsync(dst, dOut, sizeof(double) * N * N, cudaMemcpyDeviceToHost, h->stream));
    LB_CUDA(cudaStreamSynchronize(h->stream));
    LB_CUDA(cudaGetLastError());
    return LB_OK;
}

// The copy constructor KernelLFOptimization relies on (model/gp/kernel_lf_opt.hpp:79).  Nothing is copied: the clone
// references the source's buffers, and whichever of the two writes first (lb_fit, lb_append, lb_set_data, ...) takes a
// private buffer from the pool at that point (make_unique).  K^-1 / L^-1 are not carried over (the reference's copy
// keeps _inv_kernel, but every consumer recomputes it after recompute(), and lb_compute_inv_kernel rebuilds it on demand).
int lb_clone(const lb_gp* src, lb_gp** out)
{
    if (!src || !out) return LB_ERR_ARG;
    LB_DEVICE(src);
    lb_gp* h = nullptr;
    int rc = lb_create(&h, src->device, src->precision);
    if (rc) return rc;
    // pending writes of the source (e.g. lb_fit_async) must be complete before another stream reads the shared buffers
    if (cudaStreamSynchronize(src->stream) != cudaSuccess) { lb_destroy(h); return LB_ERR_CUDA; }
    h->kp = src->kp; h->kernel_set = src->kernel_set; h->n_hparams = src->n_hparams;
    h->N = src->N; h->D = src->D; h->P = src->P;
    h->kp.lambda = nullptr;
    std::memcpy(full(h)->ex.lambda_host, full(src)->ex.lambda_host, sizeof(full(h)->ex.lambda_host));
    if (src->kp.klam > 0) { // own copy of the Lambda matrix (rewritten by every lb_set_kernel)
        if (lb_dalloc(h, &h->dLambda, sizeof(double) * LB_MAX_D * LB_MAX_LAMBDA)
            || cudaMemcpyAsync(h->dLambda, src->dLambda, sizeof(double) * LB_MAX_D * LB_MAX_LAMBDA, cudaMemcpyDeviceToDevice, h->stream) != cudaSuccess) {
            lb_destroy(h);
            return LB_ERR_CUDA;
        }
        h->kp.lambda = h->dLambda;
    }
    if (src->Np > 0) {
        h->Np = src->Np;
        auto share = [](double* p) { lb_pool_retain(p); return p; };
        h->dX = share(src->dX);
        h->dY = share(src->dY);
        h->dXs = share(src->dXs);
        if (src->fitted) {
            h->dAlpha = share(src->dAlpha);
            h->dL = share(src->dL);
            h->dInvD = share(src->dInvD);
            h->fitted = true;
            if (src->ldig_valid) { // digit planes of the shared factor (the panel query's int8 update)
                lb_pool_retain(src->dLdig);
                h->dLdig = src->dLdig; h->ldig_np = src->ldig_np; h->ldig_valid = true;
            }
        }
        if (src->dFlags && lb_dalloc(h, &h->dFlags, sizeof(int) * (src->Np / LB_TILE + 8))) { lb_destroy(h); return LB_ERR_ALLOC; }
    }
    *out = h;
    return LB_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// Distributed fit (limbo_b200/dist_fit.py): the factor of ONE GP is computed by all ranks together with the block-cyclic
// panel factorisation of config 5 (potrf.cu lb_dchol_*), and every rank assembles the complete factor in its own handle
// from the panels that travel anyway, so that prediction / acquisition can then shard over the ranks without any further
// exchange.  The panel message of pair p is  [ head: the pair's 256 x 256 diagonal block, column-major ld 256 |
// inv(L_kk), inv(L_k+1,k+1) : 2 x 128 x 128 | rows below the pair, ld = Nd - (kpair + 2) * 128 ]  (LB_DCHOL_HEAD doubles
// before the rows).  The update order per tile is lb_fit's, so the assembled factor is bit-identical to lb_fit's.
// ---------------------------------------------------------------------------------------------------------------------
#define LB_DCHOL_HEAD (2 * LB_TILE * 2 * LB_TILE + 2 * LB_TILE * LB_TILE)

namespace {
// head of the message from the owner's pair columns (dCols: Nd x 256, ld = Nd) and its two diagonal-block inverses
__global__ void __launch_bounds__(256)
dchol_pack_head_kernel(const double* __restrict__ cols, int64_t ld, int64_t row0, const double* __restrict__ invD, double* __restrict__ head)
{
    const int idx = blockIdx.x * 256 + threadIdx.x;
    constexpr int DIAG = 2 * LB_TILE * 2 * LB_TILE;
    if (idx < DIAG) {
        const int r = idx & 255, c = idx >> 8;
        head[idx] = cols[row0 + r + (int64_t)c * ld];
    }
    else if (idx < LB_DCHOL_HEAD)
        head[idx] = invD[idx - DIAG];
}
// message -> this rank's factor storage: L[row0 + r, row0 + c] (r < 256: head; r >= 256: rows below), invD[kpair], invD[kpair + 1]
__global__ void __launch_bounds__(256)
dchol_unpack_kernel(const double* __restrict__ msg, int64_t ldp, double* __restrict__ L, int64_t ld, int64_t row0, double* __restrict__ invD_pair)
{
    const int64_t r = (int64_t)blockIdx.x * 256 + threadIdx.x; // row inside the column block, 0 .. 256 + ldp
    const int c = blockIdx.y;
    constexpr int DIAG = 2 * LB_TILE * 2 * LB_TILE;
    if (r < 2 * LB_TILE) L[row0 + r + (row0 + c) * ld] = msg[r + c * 2 * LB_TILE];
    else if (r < 2 * LB_TILE + ldp) L[row0 + r + (row0 + c) * ld] = msg[LB_DCHOL_HEAD + (r - 2 * LB_TILE) + (int64_t)c * ldp];
    if (blockIdx.x == 0) { // the two inverse blocks: 32768 doubles over 256 columns x 256 threads
        const int idx = c * 256 + threadIdx.x;
        if (idx < 2 * LB_TILE * LB_TILE) invD_pair[idx] = msg[DIAG + idx];
    }
}
} // namespace

// the owner of pair `kpair`: writes the head of the message (after lb_dchol_panel has factored the pair; same stream)
int lb_dchol_pack_head(lb_gp* h, const double* dCols, int64_t Nd, int kpair, const double* dInvD, double* dMsg)
{
    if (!h || !dCols || !dInvD || !dMsg) return LB_ERR_ARG;
    LB_DEVICE(h);
    dchol_pack_head_kernel<<<(LB_DCHOL_HEAD + 255) / 256, 256, 0, h->stream>>>(dCols, Nd, (int64_t)kpair * LB_TILE, dInvD, dMsg);
    h->launches++;
    LB_CUDA(cudaGetLastError());
    return LB_OK;
}

// Target handle (data and kernel already set, lb_set_data + lb_set_kernel): private factor buffers, staged samples.  The padded
// order of the handle must equal the distributed order Nd (N a multiple of 256, or 128 < N mod 256).
int lb_dchol_adopt_begin(lb_gp* h, int64_t Nd)
{
    if (!h) return LB_ERR_ARG;
    if (!h->kernel_set || h->N == 0 || h->Np == 0 || !h->dX) return LB_ERR_STATE;
    if (h->Np != Nd) return LB_ERR_UNSUPPORTED;
    LB_DEVICE(h);
    int rc;
    if ((rc = ensure_fit_buffers(h))) return rc;
    if ((rc = lb_launch_scale_x(h))) return rc;
    LB_CUDA(cudaMemsetAsync(h->dInfo, 0, 2 * sizeof(int), h->stream));
    h->fitted = false; h->linv_valid = false; h->linv_levels = 0; h->ldig_valid = false; h->kinv_valid = false; h->linv32_valid = false;
    return LB_OK;
}
// one received (or own) panel message into the handle's L / invD, on `stream` (cudaStream_t as void*; NULL = the handle's)
int lb_dchol_unpack(lb_gp* h, const double* dMsg, int64_t Nd, int kpair, void* stream)
{
    if (!h || !dMsg || !h->dL || !h->dInvD || h->Np != Nd) return LB_ERR_ARG;
    LB_DEVICE(h);
    const int64_t row0 = (int64_t)kpair * LB_TILE, ldp = Nd - row0 - 2 * LB_TILE;
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    dim3 grid((unsigned)((2 * LB_TILE + ldp + 255) / 256), 2 * LB_TILE);
    dchol_unpack_kernel<<<grid, 256, 0, st>>>(dMsg, ldp, h->dL, Nd, row0, h->dInvD + (int64_t)kpair * LB_TILE * LB_TILE);
    h->launches++;
    LB_CUDA(cudaGetLastError());
    return LB_OK;
}
// all panels are in: the handle is fitted (info = the distributed factorisation's), alpha is solved locally (gp.hpp:605-611)
int lb_dchol_adopt_end(lb_gp* h, int info)
{
    if (!h) return LB_ERR_ARG;
    LB_DEVICE(h);
    if (info > 0) return info;
    h->fitted = true; h->linv_valid = false; h->linv_levels = 0; h->ldig_valid = false; h->kinv_valid = false; h->linv32_valid = false;
    int rc = lb_launch_solve_alpha(h);
    if (rc) return rc;
    return check_info(h);
}

// ---- inversion of the factor spread over G GPUs, for the reduced-precision candidate path (limbo_b200_dist.h) --------------------

static int dinv_check(const lb_gp* h, int rank, int G)
{
    if (!h || G < 1 || rank < 0 || rank >= G) return LB_ERR_ARG;
    if (!h->fitted || h->N == 0) return LB_ERR_STATE;
    if (h->precision != LB_PREC_TF32 && h->precision != LB_PREC_FP16 && h->precision != LB_PREC_FP16X3) return LB_ERR_UNSUPPORTED;
    return LB_OK;
}

long long lb_dinv_chunk_bytes(const lb_gp* h, int G)
{
    int rc = dinv_check(h, 0, G);
    return rc ? (long long)rc : (long long)lb_dinv_chunk_bytes_impl(h, G);
}

int lb_dinv_columns(lb_gp* hc, int rank, int G, double* absmax_host)
{
    int rc = dinv_check(hc, rank, G);
    if (rc) return rc;
    if (!absmax_host) return LB_ERR_ARG;
    lb_gp_full* h = full(hc);
    LB_DEVICE(h);
    std::lock_guard<std::mutex> lock(h->ex.qmutex);
    QueryWs& w = h->ex.ws;
    if ((rc = ensure(h, &w.dV, &w.v_bytes, sizeof(double) * lb_linv_columns_scratch_doubles(h, G)))) return rc;
    if ((rc = lb_launch_linv_columns(h, h->stream, rank, G, w.dV, &h->launches))) return rc;
    return lb_dinv_absmax(h, w.dV, G, absmax_host);
}

int lb_dinv_pack(lb_gp* hc, int rank, int G, double absmax_all, void* dChunk)
{
    int rc = dinv_check(hc, rank, G);
    if (rc) return rc;
    if (!dChunk) return LB_ERR_ARG;
    lb_gp_full* h = full(hc);
    LB_DEVICE(h);
    std::lock_guard<std::mutex> lock(h->ex.qmutex);
    QueryWs& w = h->ex.ws;
    if (!w.dV || w.v_bytes < sizeof(double) * lb_linv_columns_scratch_doubles(h, G)) return LB_ERR_STATE; // lb_dinv_columns first
    return lb_dinv_pack_impl(h, w.dV, rank, G, absmax_all, dChunk);
}

int lb_dinv_adopt(lb_gp* hc, int G, const void* dAll, double absmax_all)
{
    int rc = dinv_check(hc, 0, G);
    if (rc) return rc;
    if (!dAll) return LB_ERR_ARG;
    lb_gp_full* h = full(hc);
    LB_DEVICE(h);
    std::lock_guard<std::mutex> lock(h->ex.qmutex);
    return lb_dinv_adopt_impl(h, G, dAll, absmax_all);
}

// per-kernel-class event timing for bench.py's roofline (not part of the reference-facing header)
int lb_profile_enable(lb_gp* h, int on)
{
    if (!h) return LB_ERR_ARG;
    LB_DEVICE(h);
    if (on && !h->prof) h->prof = new Profiler();
    if (!on && h->prof) {
        cudaStreamSynchronize(h->stream);
        Profiler* p = (Profiler*)h->prof;
        for (auto& r : p->recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
        for (auto e : p->pool) cudaEventDestroy(e);
        delete p;
        h->prof = nullptr;
    }
    return LB_OK;
}
// accumulates finished records; ms_out / count_out have LB_PC_COUNT entries; reset != 0 clears the totals
int lb_profile_read(lb_gp* h, double* ms_out, long long* count_out, int reset)
{
    if (!h || !h->prof) return LB_ERR_STATE;
    LB_DEVICE(h);
    Profiler* p = (Profiler*)h->prof;
    LB_CUDA(cudaStreamSynchronize(h->stream));
    std::lock_guard<std::mutex> lk(p->mu);
    const bool dump = getenv("LB_PROF_TIMELINE") != nullptr; // debug: per-launch (class, start, end) in ms from the first record
    for (auto& r : p->recs) {
        float ms = 0.f;
        if (dump && !p->recs.empty()) {
            float t0 = 0.f, t1 = 0.f;
            if (cudaEventElapsedTime(&t0, p->recs[0].a, r.a) == cudaSuccess && cudaEventElapsedTime(&t1, p->recs[0].a, r.b) == cudaSuccess)
                fprintf(stderr, "LBTL %d %.3f %.3f\n", r.cls, t0, t1);
        }
        if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) { p->ms[r.cls] += ms; p->n[r.cls]++; }
        p->pool.push_back(r.a); p->pool.push_back(r.b);
    }
    p->recs.clear();
    for (int c = 0; c < LB_PC_COUNT; ++c) {
        if (ms_out) ms_out[c] = p->ms[c];
        if (count_out) count_out[c] = p->n[c];
        if (reset) { p->ms[c] = 0; p->n[c] = 0; }
    }
    return LB_OK;
}

const char* lb_strerror(int code)
{
    if (code > 0) return "kernel matrix is not positive definite (value = 1-based index of the failing pivot)";
    switch (code) {
    case LB_OK: return "ok";
    case LB_ERR_ARG: return "invalid argument";
    case LB_ERR_CUDA: return "CUDA runtime error (see lb_last_cuda_error)";
    case LB_ERR_STATE: return "call sequence error (data / kernel / fit missing)";
    case LB_ERR_ALLOC: return "device memory allocation failed";
    case LB_ERR_UNSUPPORTED: return "unsupported kernel / acquisition / precision";
    case LB_ERR_TIMEOUT: return "device-side wait timed out";
    default: return "unknown error";
    }
}

const char* lb_last_cuda_error(void) { return g_last_cuda_error.c_str(); }

} // extern "C"
