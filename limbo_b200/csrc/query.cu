// limbo_b200/csrc/query.cu — batched GP prediction and acquisition.
//
// Replaces, for a batch of M candidates at once, the one-point-at-a-time
//   GP::_compute_k (model/gp.hpp:626-632)   -> kstar_kernel      (K* = k(X, Xq), N x M)
//   GP::_mu        (model/gp.hpp:613-616)   -> mu_kernel         (K*^T alpha)
//   GP::_sigma     (model/gp.hpp:618-624)   -> query_step_kernel (V = L^-1 K*, blocked TRSM on DMMA)
//                                              + colnorm_kernel  (k(v,v) - |V_m|^2, clamp, + noise gp.hpp:166)
//   acqui::UCB / GP_UCB / EI (acqui/ucb.hpp:83-90, gp_ucb.hpp:96-103, ei.hpp:85-116)
//                                           -> acq_kernel + argmax reduction
#include "gemm.cuh"
#include <cfloat>
#include <cstdlib>

namespace {

constexpr int DCH = 16;

// K*[n, m] = k(x_n, q_m), no noise (kernel.hpp:81-84 with i=-1, j=-2).
// grid: (Np/128, Mp/128); V is Np x Mp column-major (ld = Np).
__global__ void __launch_bounds__(256, 2)
kstar_kernel(const double* __restrict__ Xs, int64_t Np, int64_t N, const double* __restrict__ Qs, int64_t Mp,
    int64_t M, double* __restrict__ V, KernParams kp)
{
    __shared__ __align__(128) double sxi[DCH][LB_TILE];
    __shared__ __align__(128) double sxj[DCH][LB_TILE];
    __shared__ __align__(8) uint64_t bar;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int li = lane & 7, lj = lane >> 3;
    const int D = kp.D;
    const int64_t i0 = (int64_t)blockIdx.x * LB_TILE, j0 = (int64_t)blockIdx.y * LB_TILE;
    const int r0 = warp * 16 + 2 * li;
    if (tid == 0) {
        lb_mbar_init(&bar, 1);
        lb_fence_barrier_init();
    }
    __syncthreads();
    uint32_t phase = 0;
    const int npass = (D + DCH - 1) / DCH;
    for (int h = 0; h < 2; ++h) {
        double z[8][4];
#pragma unroll
        for (int c = 0; c < 8; ++c)
#pragma unroll
            for (int e = 0; e < 4; ++e) z[c][e] = 0.0;
        for (int pass = 0; pass < npass; ++pass) {
            const int d0 = pass * DCH;
            const int dc = min(DCH, D - d0);
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
                lb_mbar_wait(&bar, phase);
                phase ^= 1;
            }
            for (int d = 0; d < dc; ++d) {
                const double2 xi = *reinterpret_cast<const double2*>(&sxi[d][r0]);
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const double2 xj = *reinterpret_cast<const double2*>(&sxj[d][h * 64 + c * 8 + 2 * lj]);
                    double q;
                    q = xi.x - xj.x; z[c][0] = fma(q, q, z[c][0]);
                    q = xi.y - xj.x; z[c][1] = fma(q, q, z[c][1]);
                    q = xi.x - xj.y; z[c][2] = fma(q, q, z[c][2]);
                    q = xi.y - xj.y; z[c][3] = fma(q, q, z[c][3]);
                }
            }
        }
        const int64_t gi = i0 + r0;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const int64_t gj = j0 + h * 64 + c * 8 + 2 * lj;
            double v[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int64_t ii = gi + (e & 1), jj = gj + (e >> 1);
                double k = lb_kernel_from_z(kp.id, z[c][e], kp);
                if (ii >= N || jj >= M) k = 0.0;
                v[e] = k;
            }
            *reinterpret_cast<double2*>(&V[gi + gj * Np]) = make_double2(v[0], v[1]);
            *reinterpret_cast<double2*>(&V[gi + (gj + 1) * Np]) = make_double2(v[2], v[3]);
        }
    }
}

// mu[m*P + p] = sum_n K*[n,m] alpha[n,p]   (one CTA per candidate, fixed order -> deterministic)
__global__ void __launch_bounds__(256)
mu_kernel(const double* __restrict__ V, int64_t Np, const double* __restrict__ alpha, int P, double* __restrict__ mu)
{
    __shared__ double red[8];
    const int64_t m = blockIdx.x;
    const double* col = V + m * Np;
    for (int p = 0; p < P; ++p) {
        const double* a = alpha + (int64_t)p * Np;
        double s = 0.0;
        for (int64_t n = threadIdx.x; n < Np; n += 256) s = fma(col[n], a[n], s);
        s = lb_warp_sum(s);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int w = 0; w < 8; ++w) t += red[w];
            mu[m * P + p] = t;
        }
        __syncthreads();
    }
}

// One block-row step of V <- L^-1 V:
//   V_i <- inv(L_ii) * (V_i - L[i, 0:i] V[0:i])          grid = Mp / BN
template <typename C>
__global__ void __launch_bounds__(C::THREADS, 1)
query_step_kernel(const double* __restrict__ L, int64_t ld, const double* __restrict__ invD, double* __restrict__ V,
    int i)
{
    extern __shared__ __align__(16) double smem[];
    constexpr int PB = lbg::BM + 4;
    double* sT = smem + C::A_PIPE_DOUBLES; // overlays the B pipeline stages
    const int64_t col0 = (int64_t)blockIdx.x * C::BN;
    double* Vc = V + col0 * ld;
    lbg::Acc<C> acc;
    double* Vi = Vc + (int64_t)i * LB_TILE;
    lbg::load_acc<C>(acc, Vi, ld); // acc = V_i, then acc -= L[i,0:i] V[0:i]
    if (i > 0) lbg::mainloop<C, false, true, true>(acc, L + (int64_t)i * LB_TILE, ld, Vc, ld, i * LB_TILE, smem);
    // t -> smem [n][k]
    lbg::for_each_acc<C>(acc, [&](int r, int c, double& v) { sT[c * PB + r] = v; });
    __syncthreads();
    lbg::Acc<C> acc2;
    acc2.zero();
    lbg::mainloop_resB<C>(acc2, invD + (int64_t)i * LB_TILE * LB_TILE, LB_TILE, sT, smem);
    lbg::store_acc<C>(acc2, Vi, ld);
}

// sigma2[m] = k(v,v) - |V_m|^2, clamped (gp.hpp:623), + noise (gp.hpp:166)
__global__ void __launch_bounds__(256)
colnorm_kernel(const double* __restrict__ V, int64_t Np, double kvv, double noise, double* __restrict__ s2)
{
    __shared__ double red[8];
    const int64_t m = blockIdx.x;
    const double* col = V + m * Np;
    double s = 0.0;
    for (int64_t n = threadIdx.x; n < Np; n += 256) { double v = col[n]; s = fma(v, v, s); }
    s = lb_warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += red[w];
        double res = kvv - t;
        res = (res <= DBL_EPSILON) ? 0.0 : res;
        s2[m] = res + noise;
    }
}

// acquisition value per candidate (FirstElem aggregator, bo_base.hpp:99-105)
//   acq_id 0: UCB / GP_UCB  mu + p0 * sqrt(s2)                 ucb.hpp:89, gp_ucb.hpp:102
//   acq_id 1: EI  (p0 = f_max, p1 = jitter)                    ei.hpp:92-115
__device__ __forceinline__ double acq_value(int acq_id, double mu, double s2, double p0, double p1)
{
    if (acq_id == 0) return mu + p0 * sqrt(s2);
    double sigma = sqrt(s2);
    if (sigma < 1e-10) return 0.0;
    double X = mu - p0 - p1;
    double Z = X / sigma;
    double phi = exp(-0.5 * (Z * Z)) / sqrt(2.0 * M_PI);
    double Phi = 0.5 * erfc(-Z / sqrt(2.0));
    return X * Phi + sigma * phi;
}

__global__ void __launch_bounds__(256)
acq_kernel(int acq_id, double p0, double p1, int64_t M, const double* __restrict__ mu0, int mu_stride,
    const double* __restrict__ mean_at_q, double mean_const, const double* __restrict__ s2, double* __restrict__ acq,
    double* __restrict__ blk_val, long long* __restrict__ blk_idx)
{
    __shared__ double sv[256];
    __shared__ long long si[256];
    int64_t m = blockIdx.x * (int64_t)256 + threadIdx.x;
    double v = -DBL_MAX;
    long long idx = LLONG_MAX;
    if (m < M) {
        double mu = mu0[m * mu_stride] + (mean_at_q ? mean_at_q[m] : mean_const);
        v = acq_value(acq_id, mu, s2[m], p0, p1);
        if (acq) acq[m] = v;
        idx = m;
        if (!(v == v)) { v = -DBL_MAX; } // NaN never wins
    }
    sv[threadIdx.x] = v;
    si[threadIdx.x] = idx;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            double v2 = sv[threadIdx.x + o];
            long long i2 = si[threadIdx.x + o];
            if (v2 > sv[threadIdx.x] || (v2 == sv[threadIdx.x] && i2 < si[threadIdx.x])) {
                sv[threadIdx.x] = v2;
                si[threadIdx.x] = i2;
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        blk_val[blockIdx.x] = sv[0];
        blk_idx[blockIdx.x] = si[0];
    }
}

__global__ void __launch_bounds__(256)
argmax_final_kernel(int nblk, const double* __restrict__ blk_val, const long long* __restrict__ blk_idx,
    double* __restrict__ best_val, long long* __restrict__ best_idx)
{
    __shared__ double sv[256];
    __shared__ long long si[256];
    double v = -DBL_MAX;
    long long idx = LLONG_MAX;
    for (int b = threadIdx.x; b < nblk; b += 256) {
        double v2 = blk_val[b];
        long long i2 = blk_idx[b];
        if (v2 > v || (v2 == v && i2 < idx)) { v = v2; idx = i2; }
    }
    sv[threadIdx.x] = v;
    si[threadIdx.x] = idx;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            double v2 = sv[threadIdx.x + o];
            long long i2 = si[threadIdx.x + o];
            if (v2 > sv[threadIdx.x] || (v2 == sv[threadIdx.x] && i2 < si[threadIdx.x])) {
                sv[threadIdx.x] = v2;
                si[threadIdx.x] = i2;
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        *best_val = sv[0];
        *best_idx = si[0];
    }
}

using StepCfg = lbg::CfgStep;
constexpr size_t step_smem()
{
    constexpr size_t a = (size_t)StepCfg::A_PIPE_DOUBLES * sizeof(double);
    constexpr size_t b = (size_t)lbg::STAGES * StepCfg::B_STAGE * sizeof(double);
    constexpr size_t t = (size_t)StepCfg::BN * (lbg::BM + 4) * sizeof(double);
    return a + (t > b ? t : b);
}

LbOncePerDevice g_attr_once;
int set_attrs()
{
    if (!g_attr_once.need()) return LB_OK;
    LB_CUDA(cudaFuncSetAttribute(query_step_kernel<StepCfg>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)step_smem()));
    return LB_OK;
}

} // namespace

// Blocked V <- L^-1 V for a Np x Mp right-hand side (also used by K^-1).
int lb_launch_trsm_lower(const lb_gp* h, cudaStream_t st, double* dV, int64_t Mp, int i_begin, long long* launches)
{
    int rc = set_attrs();
    if (rc) return rc;
    const int T = (int)(h->Np / LB_TILE);
    LbProfScope ps(h, st, LB_PC_QSTEP);
    for (int i = i_begin; i < T; ++i) {
        query_step_kernel<StepCfg><<<(unsigned)(Mp / StepCfg::BN), StepCfg::THREADS, step_smem(), st>>>(h->dL, h->Np, h->dInvD, dV, i);
        if (launches) ++*launches;
    }
    LB_CUDA(cudaGetLastError());
    return LB_OK;
}

int lb_launch_query(const lb_gp* h, cudaStream_t st, int64_t M, const double* dQs, int64_t Mp, double* dV, double* dMu,
    double* dS2, long long* launches)
{
    dim3 grid((unsigned)(h->Np / LB_TILE), (unsigned)(Mp / LB_TILE));
    {
        LbProfScope ps(h, st, LB_PC_KSTAR);
        kstar_kernel<<<grid, 256, 0, st>>>(h->dXs, h->Np, h->N, dQs, Mp, M, dV, h->kp);
    }
    {
        LbProfScope ps(h, st, LB_PC_QREDUCE);
        mu_kernel<<<(unsigned)M, 256, 0, st>>>(dV, h->Np, h->dAlpha, h->P, dMu);
    }
    if (launches) *launches += 2;
    int rc = lb_launch_trsm_lower(h, st, dV, Mp, 0, launches);
    if (rc) return rc;
    const double kvv = h->kp.sf2; // every kernel here has k(v,v) = sigma_f^2
    {
        LbProfScope ps(h, st, LB_PC_QREDUCE);
        colnorm_kernel<<<(unsigned)M, 256, 0, st>>>(dV, h->Np, kvv, h->kp.noise, dS2);
    }
    if (launches) ++*launches;
    LB_CUDA(cudaGetLastError());
    return LB_OK;
}

int lb_launch_acq_full(cudaStream_t st, int acq_id, double p0, double p1, int64_t M, const double* dMu, int mu_stride,
    const double* dMeanAtQ, double mean_const, const double* dS2, double* dAcq, double* dBlkVal, long long* dBlkIdx,
    double* dBestVal, long long* dBestIdx, long long* launches)
{
    const int nblk = (int)((M + 255) / 256);
    acq_kernel<<<nblk, 256, 0, st>>>(acq_id, p0, p1, M, dMu, mu_stride, dMeanAtQ, mean_const, dS2, dAcq, dBlkVal, dBlkIdx);
    argmax_final_kernel<<<1, 256, 0, st>>>(nblk, dBlkVal, dBlkIdx, dBestVal, dBestIdx);
    if (launches) *launches += 2;
    LB_CUDA(cudaGetLastError());
    return LB_OK;
}

// ===========================================================================
// Fused, persistent batched query (the production path for D <= 16, P <= 4).
//
// One CTA per candidate slab of up to 72 candidates; the slab walks all T row
// blocks of the factor by itself, so there is no inter-CTA dependency, no
// per-step launch and no wave quantisation (slabs are sized so that all 148 SMs
// get 8 or 9 n8-tiles).  For row block i:
//   acc  = K*[i, slab]  (generated on chip from X_i and the slab's candidates;
//                        mu += K*^T alpha on the way)
//   acc -= L[i, 0:i] V[0:i, slab]      (DMMA, A = L via L2, B = the CTA's private V)
//   V_i  = inv(L_ii) acc               (DMMA), |V_i|^2 accumulated per candidate
// The 16 warps are 8 row-warps x 2 K-groups: group g takes the g-th k8 step of
// every 16-deep pipeline stage and the two partial tiles are combined through
// shared memory once per row block, which keeps 4 DMMA-issuing warps on every
// SM sub-partition.
// ===========================================================================
namespace slab {

constexpr int NTMAX = 9;
constexpr int SLAB = NTMAX * 8;  // 72
constexpr int THREADS = 512;
constexpr int BK = 32;
constexpr int STAGES = 3;
constexpr int PA = 132;  // A stage [32][132]
constexpr int PBK = 36;  // B stage [SLAB][36]
constexpr int PT = 132;  // resident tile [SLAB][132]
constexpr int DMAXF = 16;
constexpr int PMAXF = 4;
constexpr int A_STAGE = BK * PA;     // 2112
constexpr int B_STAGE = SLAB * PBK;  // 1440
constexpr int OFF_A = 0;
constexpr int OFF_B = OFF_A + STAGES * A_STAGE;
constexpr int OFF_T = OFF_B; // the resident tile overlays the B stages (never live at the same time)
constexpr int BT_DOUBLES = (STAGES * B_STAGE > SLAB * PT) ? STAGES * B_STAGE : SLAB * PT;
constexpr int OFF_X = OFF_B + BT_DOUBLES;
constexpr int OFF_Q = OFF_X + DMAXF * LB_TILE;
constexpr int OFF_AL = OFF_Q + DMAXF * SLAB;
constexpr int OFF_RED = OFF_AL + PMAXF * LB_TILE;
constexpr int OFF_MU = OFF_RED + 8 * SLAB;
constexpr int OFF_NRM = OFF_MU + PMAXF * SLAB;
constexpr int SMEM_DOUBLES = OFF_NRM + SLAB;
constexpr size_t SMEM_BYTES = (size_t)SMEM_DOUBLES * sizeof(double);

// per-thread copy plans (chunk -> offsets computed once, see gemm.cuh TilePlan)
struct PlanA { // 32 k-columns x 128 rows, outer-contiguous: 2048 chunks, 4 per thread
    int goff[4];
    int soff[4];
    __device__ __forceinline__ void init(int ld)
    {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int c = threadIdx.x + q * THREADS;
            const int k = c >> 6, oc = c & 63;
            goff[q] = k * ld + 2 * oc;
            soff[q] = k * PA + 2 * oc;
        }
    }
    __device__ __forceinline__ void issue(double* s, const double* __restrict__ g) const
    {
#pragma unroll
        for (int q = 0; q < 4; ++q) lb_cp_async16(s + soff[q], g + goff[q]);
    }
};
struct PlanB { // ncols candidates x 32 k, k-contiguous: ncols * 16 (<= 1152) chunks, up to 3 per thread
    int goff[3];
    int soff[3];
    __device__ __forceinline__ void init(int ld)
    {
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            const int c = threadIdx.x + q * THREADS;
            const int n = c >> 4, kc = c & 15;
            goff[q] = n * ld + 2 * kc;
            soff[q] = n * PBK + 2 * kc;
        }
    }
    __device__ __forceinline__ void issue(double* s, const double* __restrict__ g, int ncols) const
    {
#pragma unroll
        for (int q = 0; q < 3; ++q)
            if ((int)threadIdx.x + q * THREADS < ncols * 16) lb_cp_async16(s + soff[q], g + goff[q]);
    }
};

// 32 k-columns of a 128 x 128 inverse diagonal block (ld = 128); offsets recomputed on the fly (4 stages per row block)
__device__ __forceinline__ void issue_invd_stage(double* s, const double* __restrict__ g)
{
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int c = threadIdx.x + q * THREADS;
        const int k = c >> 6, oc = c & 63;
        lb_cp_async16(s + k * PA + 2 * oc, g + k * LB_TILE + 2 * oc);
    }
}

// NTC > 0: the slab width (in n8 tiles) is a compile-time constant (no predicated DMMAs); NTC == 0: runtime width.
template <int NTC>
__device__ __forceinline__ void slab_body(double* sm, const double* __restrict__ L, int64_t ld, const double* __restrict__ invD,
    const double* __restrict__ Xs, int64_t N, const double* __restrict__ Qs, int64_t Mp, int64_t M,
    const double* __restrict__ alpha, int P, const KernParams& kp, double* __restrict__ V, int64_t t0, int ntc_rt,
    double* __restrict__ mu_out, double* __restrict__ s2_out)
{
    double* sA = sm + OFF_A;
    double* sB = sm + OFF_B;
    double* sT = sm + OFF_T;
    double* sX = sm + OFF_X;
    double* sQ = sm + OFF_Q;
    double* sAl = sm + OFF_AL;
    double* sRed = sm + OFF_RED;
    double* sMu = sm + OFF_MU;
    double* sNrm = sm + OFF_NRM;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int grp = warp >> 3, wr = warp & 7;
    const int T = (int)(ld / LB_TILE);
    const int D = kp.D;
    const int r_lo = 16 * wr + g; // rows r_lo, r_lo + 8 of the current row block
    PlanA pA;
    PlanB pB;
    pA.init((int)ld);
    pB.init((int)ld);

    {
        const int ntc = (NTC > 0) ? NTC : ntc_rt;
        const int ncols = ntc * 8;
        const int64_t c0 = t0 * 8; // first candidate of the slab
        __syncthreads();
        for (int idx = tid; idx < D * ncols; idx += THREADS) {
            int d = idx / ncols, c = idx - d * ncols;
            sQ[d * SLAB + c] = Qs[(int64_t)d * Mp + c0 + c];
        }
        for (int idx = tid; idx < PMAXF * SLAB; idx += THREADS) sMu[idx] = 0.0;
        if (tid < SLAB) sNrm[tid] = 0.0;
        __syncthreads();

        for (int i = 0; i < T; ++i) {
            const int64_t row0 = (int64_t)i * LB_TILE;
            // ---- stage X_i and alpha_i ----
            for (int idx = tid; idx < D * LB_TILE; idx += THREADS) {
                int d = idx >> 7, r = idx & 127;
                sX[d * LB_TILE + r] = Xs[(int64_t)d * ld + row0 + r];
            }
            for (int idx = tid; idx < P * LB_TILE; idx += THREADS) {
                int p = idx >> 7, r = idx & 127;
                sAl[p * LB_TILE + r] = alpha[(int64_t)p * ld + row0 + r];
            }
            // prefetch the first pipeline stages of phase 1 while K* is generated
            const int nk = i * (LB_TILE / BK);
            const double* gA = L + row0;          // L[i-block rows, k = 0..]
            const double* gB = V;                 // V[k = 0.., slab]
#pragma unroll
            for (int st = 0; st < STAGES - 1; ++st) {
                if (st < nk) {
                    pA.issue(sA + st * A_STAGE, gA + (int64_t)st * BK * ld);
                    pB.issue(sB + st * B_STAGE, gB + st * BK, ncols);
                }
                lb_cp_async_commit();
            }
            __syncthreads();
            // ---- phase 0: acc = K*[i, slab] (group 0), mu partials ----
            double acc[NTMAX][4];
#pragma unroll
            for (int nt = 0; nt < NTMAX; ++nt)
#pragma unroll
                for (int e = 0; e < 4; ++e) acc[nt][e] = 0.0;
            if (grp == 0) {
#pragma unroll
                for (int nt = 0; nt < NTMAX; ++nt) {
                    if (nt < ntc) {
                        double z[4] = {0.0, 0.0, 0.0, 0.0};
                        const int cl = 8 * nt + 2 * t;
                        for (int d = 0; d < D; ++d) {
                            const double x0 = sX[d * LB_TILE + r_lo], x1 = sX[d * LB_TILE + r_lo + 8];
                            const double q0 = sQ[d * SLAB + cl], q1 = sQ[d * SLAB + cl + 1];
                            double u;
                            u = x0 - q0; z[0] = fma(u, u, z[0]);
                            u = x0 - q1; z[1] = fma(u, u, z[1]);
                            u = x1 - q0; z[2] = fma(u, u, z[2]);
                            u = x1 - q1; z[3] = fma(u, u, z[3]);
                        }
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const int64_t gr = row0 + r_lo + 8 * (e >> 1), gc = c0 + cl + (e & 1);
                            double k = lb_kernel_from_z(kp.id, z[e], kp);
                            if (gr >= N || gc >= M) k = 0.0;
                            acc[nt][e] = k;
                        }
                    }
                }
            }
            // mu += K*^T alpha (deterministic: shuffle over the 8 row lanes, then a fixed-order sum over warps)
            for (int p = 0; p < P; ++p) {
                if (grp == 0) {
                    const double a0 = sAl[p * LB_TILE + r_lo], a1 = sAl[p * LB_TILE + r_lo + 8];
#pragma unroll
                    for (int nt = 0; nt < NTMAX; ++nt) {
                        if (nt < ntc) {
                            double s0 = fma(acc[nt][0], a0, acc[nt][2] * a1);
                            double s1 = fma(acc[nt][1], a0, acc[nt][3] * a1);
#pragma unroll
                            for (int o = 4; o < 32; o <<= 1) {
                                s0 += __shfl_xor_sync(0xffffffffu, s0, o);
                                s1 += __shfl_xor_sync(0xffffffffu, s1, o);
                            }
                            if (g == 0) {
                                sRed[wr * SLAB + 8 * nt + 2 * t] = s0;
                                sRed[wr * SLAB + 8 * nt + 2 * t + 1] = s1;
                            }
                        }
                    }
                }
                __syncthreads();
                if (tid < ncols) {
                    double sum = 0.0;
#pragma unroll
                    for (int w = 0; w < 8; ++w) sum += sRed[w * SLAB + tid];
                    sMu[p * SLAB + tid] += sum;
                }
                __syncthreads();
            }
            // ---- phase 1: acc -= L[i, 0:i] V[0:i] ----
            for (int kt = 0; kt < nk; ++kt) {
                lb_cp_async_wait<STAGES - 2>();
                __syncthreads();
                const double* a_s = sA + (kt % STAGES) * A_STAGE;
                const double* b_s = sB + (kt % STAGES) * B_STAGE;
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) { // the group's four k4 steps: 2 * ntc independent DMMA.8x8x4 each
                    const int k0 = 16 * grp + 4 * kk;
                    const double a0 = -a_s[(k0 + t) * PA + r_lo], a1 = -a_s[(k0 + t) * PA + r_lo + 8];
                    double b[NTMAX];
#pragma unroll
                    for (int nt = 0; nt < NTMAX; ++nt) b[nt] = (nt < ntc) ? b_s[(8 * nt + g) * PBK + k0 + t] : 0.0;
#pragma unroll
                    for (int nt = 0; nt < NTMAX; ++nt) {
                        if (nt < ntc) {
                            lb_dmma_8x8x4(acc[nt][0], acc[nt][1], a0, b[nt]);
                            lb_dmma_8x8x4(acc[nt][2], acc[nt][3], a1, b[nt]);
                        }
                    }
                }
                // prefetch slab kt+2 behind the DMMA stream (its slot was last read before this iteration's barrier)
                const int nx = kt + STAGES - 1;
                if (nx < nk) {
                    pA.issue(sA + (nx % STAGES) * A_STAGE, gA + (int64_t)nx * BK * ld);
                    pB.issue(sB + (nx % STAGES) * B_STAGE, gB + nx * BK, ncols);
                }
                lb_cp_async_commit();
            }
            lb_cp_async_wait<0>();
            __syncthreads();
            // ---- combine the two K-groups: t = acc0 + acc1 -> sT[n][k] ----
            if (grp == 1) {
#pragma unroll
                for (int nt = 0; nt < NTMAX; ++nt)
                    if (nt < ntc)
#pragma unroll
                        for (int e = 0; e < 4; ++e) sT[(8 * nt + 2 * t + (e & 1)) * PT + r_lo + 8 * (e >> 1)] = acc[nt][e];
            }
            // start streaming inv(L_ii) (phase 2 operand A) meanwhile
            const double* gD = invD + (int64_t)i * LB_TILE * LB_TILE;
#pragma unroll
            for (int st = 0; st < STAGES - 1; ++st) {
                issue_invd_stage(sA + st * A_STAGE, gD + (int64_t)st * BK * LB_TILE);
                lb_cp_async_commit();
            }
            __syncthreads();
            if (grp == 0) {
#pragma unroll
                for (int nt = 0; nt < NTMAX; ++nt)
                    if (nt < ntc)
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            double* p = &sT[(8 * nt + 2 * t + (e & 1)) * PT + r_lo + 8 * (e >> 1)];
                            *p = acc[nt][e] + *p;
                        }
            }
#pragma unroll
            for (int nt = 0; nt < NTMAX; ++nt)
#pragma unroll
                for (int e = 0; e < 4; ++e) acc[nt][e] = 0.0;
            // ---- phase 2: acc = inv(L_ii) * t ----
            for (int kt = 0; kt < LB_TILE / BK; ++kt) {
                lb_cp_async_wait<STAGES - 2>();
                __syncthreads(); // also publishes group 0's sT writes on the first iteration
                const int nx = kt + STAGES - 1;
                if (nx < LB_TILE / BK) issue_invd_stage(sA + (nx % STAGES) * A_STAGE, gD + (int64_t)nx * BK * LB_TILE);
                lb_cp_async_commit();
                const double* a_s = sA + (kt % STAGES) * A_STAGE;
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    const int k0 = 16 * grp + 4 * kk;
                    const double a0 = a_s[(k0 + t) * PA + r_lo], a1 = a_s[(k0 + t) * PA + r_lo + 8];
#pragma unroll
                    for (int nt = 0; nt < NTMAX; ++nt) {
                        if (nt < ntc) {
                            const double b = sT[(8 * nt + g) * PT + kt * BK + k0 + t];
                            lb_dmma_8x8x4(acc[nt][0], acc[nt][1], a0, b);
                            lb_dmma_8x8x4(acc[nt][2], acc[nt][3], a1, b);
                        }
                    }
                }
            }
            lb_cp_async_wait<0>();
            __syncthreads();
            if (grp == 1) {
#pragma unroll
                for (int nt = 0; nt < NTMAX; ++nt)
                    if (nt < ntc)
#pragma unroll
                        for (int e = 0; e < 4; ++e) sT[(8 * nt + 2 * t + (e & 1)) * PT + r_lo + 8 * (e >> 1)] = acc[nt][e];
            }
            __syncthreads();
            if (grp == 0) {
#pragma unroll
                for (int nt = 0; nt < NTMAX; ++nt) {
                    if (nt < ntc) {
                        double v[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const int c = 8 * nt + 2 * t + (e & 1), r = r_lo + 8 * (e >> 1);
                            v[e] = acc[nt][e] + sT[c * PT + r];
                            V[(int64_t)c * ld + row0 + r] = v[e];
                        }
                        double s0 = fma(v[0], v[0], v[2] * v[2]);
                        double s1 = fma(v[1], v[1], v[3] * v[3]);
#pragma unroll
                        for (int o = 4; o < 32; o <<= 1) {
                            s0 += __shfl_xor_sync(0xffffffffu, s0, o);
                            s1 += __shfl_xor_sync(0xffffffffu, s1, o);
                        }
                        if (g == 0) {
                            sRed[wr * SLAB + 8 * nt + 2 * t] = s0;
                            sRed[wr * SLAB + 8 * nt + 2 * t + 1] = s1;
                        }
                    }
                }
            }
            __syncthreads(); // V_i visible to the whole CTA (later cp.async reads), sRed complete
            if (tid < ncols) {
                double sum = 0.0;
#pragma unroll
                for (int w = 0; w < 8; ++w) sum += sRed[w * SLAB + tid];
                sNrm[tid] += sum;
            }
        }
        __syncthreads();
        if (tid < ncols && c0 + tid < M) {
            double res = kp.sf2 - sNrm[tid]; // k(v,v) - z.z            gp.hpp:621
            res = (res <= DBL_EPSILON) ? 0.0 : res; //                   gp.hpp:623
            s2_out[c0 + tid] = res + kp.noise; //                        gp.hpp:166
            for (int p = 0; p < P; ++p) mu_out[(c0 + tid) * P + p] = sMu[p * SLAB + tid];
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(THREADS, 1)
query_slab_kernel(const double* __restrict__ L, int64_t ld, const double* __restrict__ invD, const double* __restrict__ Xs,
    int64_t N, const double* __restrict__ Qs, int64_t Mp, int64_t M, const double* __restrict__ alpha, int P, KernParams kp,
    double* __restrict__ Vscratch, int nslabs, int64_t ntiles_total, double* __restrict__ mu_out, double* __restrict__ s2_out)
{
    extern __shared__ __align__(16) double sm[];
    double* V = Vscratch + (int64_t)blockIdx.x * ld * SLAB; // private [c][n], ld per candidate
    for (int s = blockIdx.x; s < nslabs; s += gridDim.x) {
        // balanced partition of the n8-tiles over the slabs
        const int64_t t0 = ntiles_total * s / nslabs, t1 = ntiles_total * (s + 1) / nslabs;
        const int ntc = (int)(t1 - t0);
        if (ntc == 9) slab_body<9>(sm, L, ld, invD, Xs, N, Qs, Mp, M, alpha, P, kp, V, t0, ntc, mu_out, s2_out);
        else if (ntc == 8) slab_body<8>(sm, L, ld, invD, Xs, N, Qs, Mp, M, alpha, P, kp, V, t0, ntc, mu_out, s2_out);
        else slab_body<0>(sm, L, ld, invD, Xs, N, Qs, Mp, M, alpha, P, kp, V, t0, ntc, mu_out, s2_out);
    }
}

// One point, one launch: the candidate travels in the kernel arguments (no host-to-device copy, no packing kernel) and
// mu / sigma^2 are written straight into mapped pinned host memory (no device-to-host copies): a GP::query(v) /
// mu(v) / sigma(v) call (gp.hpp:159-191 - what the reference's inner optimisers and its regression benchmark issue 10^4
// times in a row, waf_tools/benchmark_template.cpp:95-120) costs one launch and one stream synchronisation.  Same
// slab_body as the batched kernel, so the value is bit-identical to the same point inside a slab-path batch.
struct PointArg { double x[LB_MAX_D]; };

__global__ void __launch_bounds__(THREADS, 1)
query_point_kernel(const double* __restrict__ L, int64_t ld, const double* __restrict__ invD, const double* __restrict__ Xs, int64_t N,
    const __grid_constant__ PointArg q, double* __restrict__ Qs, const double* __restrict__ alpha, int P, const __grid_constant__ KernParams kp,
    double* __restrict__ Vscratch, double* __restrict__ out)
{
    extern __shared__ __align__(16) double sm[];
    for (int idx = threadIdx.x; idx < kp.D * 8; idx += THREADS) { // staged coordinates of the point in column 0 of an 8-wide tile
        const int d = idx >> 3, c = idx & 7;
        Qs[d * LB_TILE + c] = (c == 0) ? lb_staged_coord(kp, d, [&](int r) { return q.x[r]; }) : 0.0;
    }
    __threadfence_block();
    __syncthreads();
    slab_body<0>(sm, L, ld, invD, Xs, N, Qs, LB_TILE, 1, alpha, P, kp, Vscratch, 0, 1, out, out + P);
}

LbOncePerDevice g_attr_once2;

} // namespace slab

// ===========================================================================
// Panel path for large candidate batches (M >= LB_QUERY_PANEL_MIN): V = L^-1 K* as a blocked solve over super-blocks of
// SB = 16 row tiles (2048 rows), everything on the GEMM core of gemm.cuh with long K ranges:
//     update_s :  T_s   = K*_s - L[s, 0:s] V[0:s]            (SB x Mp/128 tiles of 128 x 128, K = s * 2048)
//     solve_s  :  V_s   = inv(L_ss) T_s                      (same tiles, K = (i + 1) * 128: inv(L_ss) is lower triangular)
// inv(L_ss) = the 16-tile diagonal blocks of L^-1 from the first levels of the recursive trtri (lml.cu, ~1 % of the flops of a
// fit, cached until the next fit).  Each V block is read once per SUPER-block instead of once per 128-row block: the
// fused slab kernel above streams its private V slab T/2 times (86 GB of DRAM traffic at N = 16384, M = 10^4, ncu round 1),
// this path moves ~10 GB.  mu comes from K* before the solve; |V_c|^2 is reduced per tile in the solve epilogue (fixed
// order: lanes -> warps -> tiles), so results are run-to-run deterministic and independent of the batch composition
// (a candidate's value depends only on its own column).
// ===========================================================================
namespace panel {

constexpr int SB = 16;

// Tile configuration: CfgDual (128 x 64, two CTAs per SM) by default - a launch of 16 x ctiles tiles is a few rounds of the
// machine, and with two co-resident half-width CTAs the last, partly filled round costs half as much as with CfgWide
// (128 x 128, one CTA per SM); one CTA's C-tile prologue / epilogue also hides under the other's DMMA stream.
// Tbuf[i, ct] = V[s0 + i, ct] - L[s0 + i, 0:s0] V[0:s0, ct]       grid = nrows * (Mp / BN), row tile fastest
//
// INV = true: the right-hand sides are identity columns, V = L^-1[:, column tiles c = inv_rank + t * inv_G] (the inversion of the
// factor spread over inv_G GPUs by 128-column tiles, lb_launch_linv_columns).  Column tile c is zero above row tile c: super-blocks
// above it are skipped and the K range starts at the super-block that holds it.
template <typename C, bool INV>
__global__ void __launch_bounds__(C::THREADS, (C::THREADS == 256) ? 2 : 1)
panel_update_kernel(const double* __restrict__ L, int64_t ld, const double* __restrict__ V, double* __restrict__ Tbuf, int64_t ldt, int s0,
    int nrows, int ct0, int inv_rank, int inv_G)
{
    extern __shared__ __align__(16) double smem[];
    const int i = blockIdx.x % nrows, ct = ct0 + blockIdx.x / nrows;
    int kb = 0;
    if (INV) {
        const int c = inv_rank + (ct * C::BN / LB_TILE) * inv_G;
        if (c >= s0 + nrows) return; // (also the padding slots c >= T)
        kb = c / SB * SB;
    }
    const double* Vc = V + (int64_t)ct * C::BN * ld;
    lbg::Acc<C> acc;
    lbg::load_acc<C>(acc, Vc + (int64_t)(s0 + i) * LB_TILE, ld);
    if (s0 > kb)
        lbg::mainloop<C, false, true, true>(acc, L + (int64_t)(s0 + i) * LB_TILE + (int64_t)kb * LB_TILE * ld, ld, Vc + (int64_t)kb * LB_TILE, ld,
            (s0 - kb) * LB_TILE, smem);
    lbg::store_acc<C>(acc, Tbuf + (int64_t)i * LB_TILE + (int64_t)ct * C::BN * ldt, ldt);
}

// V[s0 + i, ct] = sum_{k <= i} Linv[s0 + i, s0 + k] Tbuf[k, ct];  normpart[(s0 + i) * Mp + c] = sum over the tile's 128 rows of V^2
template <typename C, bool INV>
__global__ void __launch_bounds__(C::THREADS, (C::THREADS == 256) ? 2 : 1)
panel_solve_kernel(const double* __restrict__ Linv, int64_t ld, const double* __restrict__ Tbuf, int64_t ldt, double* __restrict__ V, int s0,
    int nrows, double* __restrict__ normpart, int64_t Mp, int ct0, int inv_rank, int inv_G)
{
    extern __shared__ __align__(16) double smem[];
    const int i = nrows - 1 - (int)(blockIdx.x % nrows), ct = ct0 + blockIdx.x / nrows; // longest K ranges first
    int k0 = 0; // first row tile of Tbuf that is not zero
    if (INV) {
        const int c = inv_rank + (ct * C::BN / LB_TILE) * inv_G;
        if (c >= s0 + nrows) return;
        if (c > s0) k0 = c - s0;
        if (i < k0) return; // rows above the column tile stay zero (the buffer is cleared before the first super-block)
    }
    lbg::Acc<C> acc;
    acc.zero();
    lbg::mainloop<C, false, true>(acc, Linv + (int64_t)(s0 + i) * LB_TILE + (int64_t)(s0 + k0) * LB_TILE * ld, ld,
        Tbuf + (int64_t)k0 * LB_TILE + (int64_t)ct * C::BN * ldt, ldt, (i + 1 - k0) * LB_TILE, smem);
    lbg::store_acc<C>(acc, V + (int64_t)(s0 + i) * LB_TILE + (int64_t)ct * C::BN * ld, ld);
    if (INV) return;
    // column norms of the tile: per thread (2 m16 tiles x 2 row halves), then the 8 row lanes, then the 4 row warps
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int wm = warp & 3, wn = warp >> 2;
    double* sRed = smem; // [4][BN]
#pragma unroll
    for (int nt = 0; nt < C::NT; ++nt)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            double sq = 0.0;
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
                sq = fma(acc.v[mt][nt][e], acc.v[mt][nt][e], sq);
                sq = fma(acc.v[mt][nt][2 + e], acc.v[mt][nt][2 + e], sq);
            }
#pragma unroll
            for (int o = 4; o < 32; o <<= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
            if (g == 0) sRed[wm * C::BN + wn * (C::BN / C::WN) + nt * 8 + 2 * t + e] = sq;
        }
    __syncthreads();
    if ((int)threadIdx.x < C::BN) {
        const double sum = ((sRed[threadIdx.x] + sRed[C::BN + threadIdx.x]) + sRed[2 * C::BN + threadIdx.x]) + sRed[3 * C::BN + threadIdx.x];
        normpart[(int64_t)(s0 + i) * Mp + (int64_t)ct * C::BN + threadIdx.x] = sum;
    }
}

// sigma2[c] = k(v,v) - sum_t normpart[t][c], clamp (gp.hpp:623), + noise (gp.hpp:166)
__global__ void __launch_bounds__(256)
panel_finish_kernel(const double* __restrict__ normpart, int T, int64_t Mp, int64_t M, double kvv, double noise, double* __restrict__ s2)
{
    const int64_t c = blockIdx.x * (int64_t)256 + threadIdx.x;
    if (c >= M) return;
    double s = 0.0;
    for (int tt = 0; tt < T; ++tt) s += normpart[(int64_t)tt * Mp + c];
    double res = kvv - s;
    res = (res <= DBL_EPSILON) ? 0.0 : res;
    s2[c] = res + noise;
}

LbOncePerDevice g_once;

} // namespace panel

int lb_ldig_prepare(lb_gp* h);
int lb_query_i8_vexp(const lb_gp* h);
int64_t lb_query_int8_max_k();
size_t lb_query_i8_vdig_bytes(int64_t Np, int64_t Mp);
int lb_launch_vdig_split(cudaStream_t st, const double* dV, int64_t ld, int64_t Mp, int64_t r0, int64_t nr, int64_t c0, int64_t nc, int ev,
    int8_t* dVdig);
int lb_launch_panel_update_i8(const lb_gp* h, cudaStream_t st, const double* dV, const int8_t* dVdig, int64_t Mp, double* dT, int64_t ldt,
    int s0, int nrows, int ct0, int n64, int ev, int* dErr);

// workspace in doubles behind dV (Np x Mp): Tbuf (SB * 128 x Mp) + norm partials (T x Mp) [+ int8 digit planes of V (7 x Np x Mp bytes)]
size_t lb_query_panel_scratch_doubles(const lb_gp* h, int64_t Mp)
{
    const int64_t T = h->Np / LB_TILE;
    const size_t vdig = lb_query_int8_mode() ? (lb_query_i8_vdig_bytes(h->Np, Mp) + 7) / 8 : 0;
    return (size_t)(h->Np * Mp + (int64_t)panel::SB * LB_TILE * Mp + T * Mp) + vdig;
}

int lb_launch_query_panel(lb_gp* h, cudaStream_t st, int64_t M, const double* dQs, int64_t Mp, double* dWork, double* dMu, double* dS2,
    int* dErr, long long* launches)
{
    using namespace panel;
    using CW = lbg::CfgWide;
    using CD = lbg::CfgDual;
    if (g_once.need()) {
        LB_CUDA(cudaFuncSetAttribute(panel_update_kernel<CW, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CW::PIPE_BYTES));
        LB_CUDA(cudaFuncSetAttribute(panel_solve_kernel<CW, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CW::PIPE_BYTES));
        LB_CUDA(cudaFuncSetAttribute(panel_update_kernel<CD, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CD::PIPE_BYTES));
        LB_CUDA(cudaFuncSetAttribute(panel_solve_kernel<CD, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CD::PIPE_BYTES));
    }
    const int T = (int)(h->Np / LB_TILE);
    const int64_t ld = h->Np, ldt = (int64_t)SB * LB_TILE;
    double* dV = dWork;
    double* dT = dV + ld * Mp;
    double* dNorm = dT + ldt * Mp;
    int rc = lb_launch_linv_levels(h, SB); // inverse of the 16-tile diagonal blocks (kept until the next fit)
    if (rc) return rc;
    // int8 digit-product update (query_i8.cu) for the super-blocks with a K range inside its exactness bound
    const bool i8 = lb_query_int8_mode() != 0;
    int8_t* dVdig = i8 ? reinterpret_cast<int8_t*>(dNorm + (int64_t)T * Mp) : nullptr;
    const int ev = i8 ? lb_query_i8_vexp(h) : 0;
    if (i8) {
        LbProfScope ps(h, st, LB_PC_QSTEP);
        if ((rc = lb_ldig_prepare(h))) return rc; // digit planes of L (kept until the next fit)
    }
    dim3 grid((unsigned)T, (unsigned)(Mp / LB_TILE));
    {
        LbProfScope ps(h, st, LB_PC_KSTAR);
        kstar_kernel<<<grid, 256, 0, st>>>(h->dXs, h->Np, h->N, dQs, Mp, M, dV, h->kp);
    }
    {
        LbProfScope ps(h, st, LB_PC_QREDUCE);
        mu_kernel<<<(unsigned)M, 256, 0, st>>>(dV, h->Np, h->dAlpha, h->P, dMu);
    }
    if (launches) *launches += 2;
    // The chain update_s -> solve_s -> update_s+1 -> ... only couples tiles of the SAME candidate column tile: the column tiles
    // are split into two groups that walk the chain on two streams, so the tail of one group's launch (a launch is 8.5 waves of
    // 148 CTAs at M = 10^4: ncu showed the tensor pipe 93 % busy while active but 80 % of the elapsed time) is filled by the
    // other group's CTAs instead of idle SMs.
    const int ctiles = (int)(Mp / LB_TILE);
    static int split_pct = -1, use_side = -1;
    if (split_pct < 0) {
        const char* e = getenv("LB_PANEL_SPLIT");   // percentage of the column tiles in the first group; 100 = one stream
        split_pct = e ? atoi(e) : 70; // measured at N = 16384, M = 10^4: one stream 85.5 ms, 50 / 60 / 70 / 80 %: 81.3 / 80.6 / 80.5 / 80.4 ms
        if (split_pct < 1 || split_pct > 100) split_pct = 100;
        const char* e2 = getenv("LB_PANEL_SIDE");   // 1: second group on the high-priority side stream instead of a normal-priority one
        use_side = (e2 && atoi(e2) != 0) ? 1 : 0;
    }
    // LB_PANEL_CFG=1: 128 x 128 tiles (CfgWide); default 128 x 64 tiles, two CTAs per SM.  Measured at N = 16384 (ms per batch,
    // Wide / Dual): M = 1250: 13.6 / 13.1, 2500: 23.1 / 21.9, 5000: 42.6 / 39.8, 10^4: 80.4 / 78.3 (same bits: the tile shape does not
    // change any element's accumulation order).
    static int cfg_mode = -1;
    if (cfg_mode < 0) { const char* e = getenv("LB_PANEL_CFG"); cfg_mode = e ? atoi(e) : 0; }
    const bool dual = cfg_mode != 1;
    const int wmul = dual ? 2 : 1; // 64-wide column tiles per 128 candidates
    // Groups of column tiles, each walking the chain on its own stream.  Large batches: two groups (split_pct / rest).  Small batches
    // (a launch of all column tiles is under ~4 rounds of the machine: M = 1250 is 320 CTAs for 296 slots, i.e. one full round and
    // one nearly empty): up to four equal groups, so that a launch is a fraction of a round and the groups, drifting apart, keep the
    // SMs full.  LB_PANEL_GROUPS=<1..4> forces the count.  Measured at N = 16384 (ms per batch, 1 / 2 / 3 / 4 groups): M = 640: 10.6 / 9.7 /
    // 8.6 / 8.3, 1250: 14.8 / 13.3 / 12.9 / 12.5, 2500: 24.2 / 22.1 / 21.3 / 20.7, 5000: 42.6 / 40.0 / 39.8 / 39.8, 10^4: 83.6 / 78.3 / 78.4 / 78.3
    // (profiles/r02_panel_groups.txt); results do not depend on the grouping (every tile's arithmetic is unchanged).
    static int force_groups = -1;
    if (force_groups < 0) { const char* e = getenv("LB_PANEL_GROUPS"); force_groups = e ? atoi(e) : 0; }
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
    const int slots = sms * (dual ? 2 : 1);
    int ngroups = 1;
    if (split_pct < 100 && ctiles >= 4) ngroups = ((int64_t)ctiles * wmul * SB < (int64_t)4 * slots) ? 4 : 2;
    if (force_groups >= 1 && force_groups <= 4) ngroups = force_groups;
    if (ngroups > ctiles) ngroups = ctiles;
    cudaStream_t sts[4] = {st, st, st, st};
    if (ngroups >= 2) {
        if (use_side && h->side && ngroups == 2) sts[1] = h->side;
        else {
            cudaStream_t* extra[3] = {&h->aux, &h->aux2, &h->aux3};
            for (int g = 1; g < ngroups; ++g) {
                if (!*extra[g - 1] && cudaStreamCreateWithFlags(extra[g - 1], cudaStreamNonBlocking) != cudaSuccess) *extra[g - 1] = nullptr;
                if (!*extra[g - 1]) { ngroups = g; break; } // no stream: fewer groups
                sts[g] = *extra[g - 1];
            }
        }
    }
    int gbeg[5] = {0, ctiles, ctiles, ctiles, ctiles}; // first column tile (128 wide) of each group
    if (ngroups == 2) {
        int split = (ctiles * split_pct + 50) / 100;
        if (split < 1) split = 1;
        if (split > ctiles - 1) split = ctiles - 1;
        gbeg[1] = split;
    }
    else
        for (int g = 1; g < ngroups; ++g) gbeg[g] = (int)((int64_t)ctiles * g / ngroups);
    gbeg[ngroups] = ctiles;
    {
        LbProfScope ps(h, st, LB_PC_QSTEP);
        if (ngroups >= 2) {
            LB_CUDA(cudaEventRecord(h->ev[0], st));
            for (int g = 1; g < ngroups; ++g) LB_CUDA(cudaStreamWaitEvent(sts[g], h->ev[0], 0));
        }
        for (int s0 = 0; s0 < T; s0 += SB) {
            const int nrows = (T - s0 < SB) ? (T - s0) : SB;
            const bool upd_i8 = i8 && s0 > 0 && (int64_t)s0 * LB_TILE <= lb_query_int8_max_k();
            for (int g = 0; g < ngroups; ++g) {
                const int c0 = gbeg[g] * wmul, nc = (gbeg[g + 1] - gbeg[g]) * wmul;
                if (nc <= 0) continue;
                if (upd_i8) {
                    const int n64 = (gbeg[g + 1] - gbeg[g]) * 2;
                    if ((rc = lb_launch_panel_update_i8(h, sts[g], dV, dVdig, Mp, dT, ldt, s0, nrows, gbeg[g] * 2, n64, ev, dErr))) return rc;
                }
                else if (dual)
                    panel_update_kernel<CD, false><<<nrows * nc, CD::THREADS, CD::PIPE_BYTES, sts[g]>>>(h->dL, ld, dV, dT, ldt, s0, nrows, c0, 0, 1);
                else
                    panel_update_kernel<CW, false><<<nrows * nc, CW::THREADS, CW::PIPE_BYTES, sts[g]>>>(h->dL, ld, dV, dT, ldt, s0, nrows, c0, 0, 1);
                if (dual)
                    panel_solve_kernel<CD, false><<<nrows * nc, CD::THREADS, CD::PIPE_BYTES, sts[g]>>>(h->dLinv, ld, dT, ldt, dV, s0, nrows, dNorm, Mp, c0, 0, 1);
                else
                    panel_solve_kernel<CW, false><<<nrows * nc, CW::THREADS, CW::PIPE_BYTES, sts[g]>>>(h->dLinv, ld, dT, ldt, dV, s0, nrows, dNorm, Mp, c0, 0, 1);
                if (launches) *launches += 2;
                if (i8 && s0 + nrows < T) { // the solved rows feed the updates of the later super-blocks
                    if ((rc = lb_launch_vdig_split(sts[g], dV, ld, Mp, (int64_t)s0 * LB_TILE, (int64_t)nrows * LB_TILE, (int64_t)gbeg[g] * LB_TILE,
                             (int64_t)(gbeg[g + 1] - gbeg[g]) * LB_TILE, ev, dVdig))) return rc;
                    if (launches) ++*launches;
                }
            }
        }
        for (int g = 1; g < ngroups; ++g) { // join (ev[1..3]; the fit's uses of these events are complete: same stream order)
            LB_CUDA(cudaEventRecord(h->ev[g], sts[g]));
            LB_CUDA(cudaStreamWaitEvent(st, h->ev[g], 0));
        }
    }
    {
        LbProfScope ps(h, st, LB_PC_QREDUCE);
        panel_finish_kernel<<<(unsigned)((M + 255) / 256), 256, 0, st>>>(dNorm, T, Mp, M, h->kp.sf2, h->kp.noise, dS2);
    }
    if (launches) ++*launches;
    LB_CUDA(cudaGetLastError());
    return LB_OK;
}

// ---- inversion of the factor spread over G GPUs by 128-column tiles (config 4 on several GPUs: every rank scores its candidates
// against all of L^-1, gp.hpp:618-624, but computes only its own columns of it) --------------------------------------------------------
// Column tile t of the work buffer (t = 0 .. nt-1, nt = ceil(T / G)) holds L^-1[:, c] for the global tile c = rank + t * G: the blocked
// solve of the panel path with identity right-hand sides, started at the super-block that holds c.  Flops: sum_c (T - c)^2 tiles,
// i.e. N^3 / (3 G) per rank up to the super-block granularity.
namespace panel {
__global__ void __launch_bounds__(128)
identity_cols_kernel(double* __restrict__ V, int64_t ld, int rank, int G, int T)
{
    const int c = rank + (int)blockIdx.x * G;
    if (c >= T) return;
    V[(int64_t)c * LB_TILE + threadIdx.x + ((int64_t)blockIdx.x * LB_TILE + threadIdx.x) * ld] = 1.0;
}
LbOncePerDevice g_once_inv;
} // namespace panel

int64_t lb_linv_columns_width(const lb_gp* h, int G) { return ((h->Np / LB_TILE + G - 1) / G) * LB_TILE; }

size_t lb_linv_columns_scratch_doubles(const lb_gp* h, int G)
{
    const int64_t Mp = lb_linv_columns_width(h, G);
    return (size_t)(h->Np * Mp + (int64_t)panel::SB * LB_TILE * Mp);
}

int lb_launch_linv_columns(lb_gp* h, cudaStream_t st, int rank, int G, double* dWork, long long* launches)
{
    using namespace panel;
    using CD = lbg::CfgDual;
    if (g_once_inv.need()) {
        LB_CUDA(cudaFuncSetAttribute(panel_update_kernel<CD, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CD::PIPE_BYTES));
        LB_CUDA(cudaFuncSetAttribute(panel_solve_kernel<CD, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CD::PIPE_BYTES));
    }
    const int T = (int)(h->Np / LB_TILE);
    const int nt = (T + G - 1) / G;
    const int64_t ld = h->Np, ldt = (int64_t)SB * LB_TILE, Mp = (int64_t)nt * LB_TILE;
    double* dV = dWork;
    double* dT = dV + ld * Mp;
    int rc = lb_launch_linv_levels(h, SB); // inverse of the 16-tile diagonal blocks, on every rank (1.2 ms at N = 16384)
    if (rc) return rc;
    LbProfScope ps(h, st, LB_PC_TRTRI);
    LB_CUDA(cudaMemsetAsync(dV, 0, sizeof(double) * (size_t)(ld * Mp), st));
    identity_cols_kernel<<<nt, 128, 0, st>>>(dV, ld, rank, G, T);
    const int nc = nt * (LB_TILE / CD::BN);
    for (int s0 = 0; s0 < T; s0 += SB) {
        const int nrows = (T - s0 < SB) ? (T - s0) : SB;
        panel_update_kernel<CD, true><<<nrows * nc, CD::THREADS, CD::PIPE_BYTES, st>>>(h->dL, ld, dV, dT, ldt, s0, nrows, 0, rank, G);
        panel_solve_kernel<CD, true><<<nrows * nc, CD::THREADS, CD::PIPE_BYTES, st>>>(h->dLinv, ld, dT, ldt, dV, s0, nrows, nullptr, Mp, 0, rank, G);
        if (launches) *launches += 2;
    }
    if (launches) *launches += 1;
    LB_CUDA(cudaGetLastError());
    return LB_OK;
}

int lb_query_fused_supported(const lb_gp* h) { return h->kp.D <= slab::DMAXF && h->P <= slab::PMAXF; }
size_t lb_query_fused_scratch_doubles(const lb_gp* h, int grid) { return (size_t)grid * h->Np * slab::SLAB; }

// one point (host coordinates x[0..D)), results in dOutMapped[0..P) = mu, [P] = sigma^2 (device alias of pinned host memory)
int lb_launch_query_point(const lb_gp* h, cudaStream_t st, const double* x_host, double* dQs, double* dVscratch, double* dOutMapped,
    long long* launches)
{
    static LbOncePerDevice once;
    if (once.need()) {
        LB_CUDA(cudaFuncSetAttribute(slab::query_point_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)slab::SMEM_BYTES));
    }
    slab::PointArg q;
    for (int d = 0; d < LB_MAX_D; ++d) q.x[d] = d < h->D ? x_host[d] : 0.0;
    LbProfScope ps(h, st, LB_PC_QSTEP);
    slab::query_point_kernel<<<1, slab::THREADS, slab::SMEM_BYTES, st>>>(h->dL, h->Np, h->dInvD, h->dXs, h->N, q, dQs, h->dAlpha, h->P, h->kp,
        dVscratch, dOutMapped);
    if (launches) ++*launches;
    LB_CUDA(cudaGetLastError());
    return LB_OK;
}

int lb_launch_query_fused(const lb_gp* h, cudaStream_t st, int64_t M, const double* dQs, int64_t Mp, double* dVscratch,
    int grid, double* dMu, double* dS2, long long* launches)
{
    if (slab::g_attr_once2.need()) {
        LB_CUDA(cudaFuncSetAttribute(slab::query_slab_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)slab::SMEM_BYTES));
    }
    const int64_t ntiles = (M + 7) / 8;
    // slabs of <= 9 n8-tiles, a multiple of the grid so every CTA gets the same number of slabs
    int64_t nslabs = (ntiles + slab::NTMAX - 1) / slab::NTMAX;
    nslabs = (nslabs + grid - 1) / grid * grid;
    if (nslabs > ntiles) nslabs = ntiles;
    LbProfScope ps(h, st, LB_PC_QSTEP);
    slab::query_slab_kernel<<<grid, slab::THREADS, slab::SMEM_BYTES, st>>>(h->dL, h->Np, h->dInvD, h->dXs, h->N, dQs, Mp, M,
        h->dAlpha, h->P, h->kp, dVscratch, (int)nslabs, ntiles, dMu, dS2);
    if (launches) ++*launches;
    LB_CUDA(cudaGetLastError());
    return LB_OK;
}
