// limbo_b200/csrc/sparsify.cu — greedy density-based sparsification, model::SparsifiedGP::_sparsify
// (src/limbo/model/sparsified_gp.hpp:126-183), as ONE persistent cooperative launch.
//
// The reference builds the N x N distance matrix and, for each of the N - max_points removals, partial-sorts every
// remaining row to find its density (the ascending sum of its D smallest distances) and removes the row of smallest
// density, lowest index on a tie.  Here a removal re-scores only the rows it can change: row i keeps the squared distance
// thr2[i] of its D-th nearest live neighbour, and removing k changes dens[i] only if k was among those D, i.e. only if
// |x_i - x_k|^2 <= thr2[i] (on equality the row is re-scored although its density cannot change).  Every other row keeps
// exactly the multiset of D smallest distances it had, so its density is bit for bit what the reference recomputes.
//
// One removal = three grid-wide phases (cooperative launch, grid.sync between them):
//   S1  every block reduces the per-block (dens, index) minima to the same k; block 0 records it and marks k dead; each
//       block appends the affected rows of its slice to a device work list (its length is unbounded: a hub point can be
//       a neighbour of many rows);
//   S2  the work list is spread over the blocks, one row per block at a time, each re-scored from scratch over the live
//       points;
//   S3  every block writes the (dens, index) minimum of its slice.
// After the last removal nothing is re-scored (with max_points == D a row could otherwise have fewer than D neighbours).
//
// Bit-level contract with the reference (DESIGN.md §6): the distance is sqrt(sum_d (x_i,d - x_j,d)^2), summed from 0 in
// order d = 0..D-1, every operation rounded on its own (the _rn intrinsics never contract), and the density adds the D
// smallest distances in ascending order starting from 0.  Candidates are ranked by the squared sum: sqrt is monotone, so
// the D smallest squared sums give the D smallest distances.  The argmin compares (dens, index) lexicographically, so the
// result does not depend on the grid size or on the order in which the work list fills.  Distances are recomputed from
// X (D x N, dimension-major) instead of stored: N x N doubles are 32 GiB at N = 65536.
#include "../../include/limbo_b200.h"
#include "common.cuh"
#include <cooperative_groups.h>
#include <algorithm>
#include <climits>
#include <vector>

namespace cg = cooperative_groups;

namespace {

constexpr int SP_THREADS = 256;
constexpr int SP_MAX_BLOCKS_PER_SM = 4;
constexpr int SP_BATCH = 4; // candidates per thread and step in score_row

struct SpState {
    const double* X; // D x N, dimension-major
    int N, D, n_remove;
    double* dens;    // density of each live row
    double* thr2;    // squared distance of each row's D-th nearest live neighbour
    int* dead;       // 1 once removed
    int* count;      // [2] work-list lengths, double-buffered by removal parity
    int* work;       // rows to re-score (N entries: every row may be affected)
    double* bval;    // per-block (dens, index) minimum
    int* bidx;
    int* rem_idx;    // removal order
    double* rem_dens; // density at removal
};

__device__ __forceinline__ double sq_dist(const double* __restrict__ X, int N, int D, const double* xi, int j)
{
    double s = 0.0;
    for (int d = 0; d < D; ++d) {
        const double t = __dsub_rn(xi[d], __ldg(X + (size_t)d * N + j));
        s = __dadd_rn(s, __dmul_rn(t, t));
    }
    return s;
}

__device__ __forceinline__ bool pair_less(double av, int ai, double bv, int bi)
{
    return av < bv || (av == bv && ai < bi);
}

// block-wide lexicographic minimum of (v, w); every thread returns the result.  red_v / red_w hold 33 entries.
__device__ __forceinline__ void block_min_pair(double& v, int& w, double* red_v, int* red_w)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, v, o);
        const int ow = __shfl_xor_sync(0xffffffffu, w, o);
        if (pair_less(ov, ow, v, w)) { v = ov; w = ow; }
    }
    if (lane == 0) { red_v[warp] = v; red_w[warp] = w; }
    __syncthreads();
    if (warp == 0) {
        v = lane < SP_THREADS / 32 ? red_v[lane] : INFINITY;
        w = lane < SP_THREADS / 32 ? red_w[lane] : INT_MAX;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, v, o);
            const int ow = __shfl_xor_sync(0xffffffffu, w, o);
            if (pair_less(ov, ow, v, w)) { v = ov; w = ow; }
        }
        if (lane == 0) { red_v[32] = v; red_w[32] = w; }
    }
    __syncthreads();
    v = red_v[32];
    w = red_w[32];
}

// dens[i] and thr2[i] over the live points j != i, computed by the whole block.  Each thread keeps the D smallest
// squared distances of its candidates in a sorted column of `list` (D x SP_THREADS); a D-round merge of the column heads
// then yields the block's D smallest in ascending order.
__device__ void score_row(const SpState& s, int i, double* list, double* sh_x, double* red_v, int* red_w)
{
    const int tid = threadIdx.x, D = s.D, N = s.N;
    __syncthreads(); // sh_x and list may still be read from the previous row
    if (tid < D) sh_x[tid] = __ldg(s.X + (size_t)tid * N + i);
    for (int r = 0; r < D; ++r) list[r * SP_THREADS + tid] = INFINITY;
    __syncthreads();
    double worst = INFINITY;
    // SP_BATCH candidates per thread and step, their loads independent of each other; excluded candidates (self, dead,
    // past N) are skipped before the insertion
    for (int j0 = tid; j0 < N; j0 += SP_BATCH * SP_THREADS) {
        int jj[SP_BATCH];
        double acc[SP_BATCH];
#pragma unroll
        for (int u = 0; u < SP_BATCH; ++u) {
            jj[u] = min(j0 + u * SP_THREADS, N - 1);
            acc[u] = 0.0;
        }
        for (int d = 0; d < D; ++d) {
            const double xd = sh_x[d];
#pragma unroll
            for (int u = 0; u < SP_BATCH; ++u) {
                const double t = __dsub_rn(xd, __ldg(s.X + (size_t)d * N + jj[u]));
                acc[u] = __dadd_rn(acc[u], __dmul_rn(t, t));
            }
        }
#pragma unroll
        for (int u = 0; u < SP_BATCH; ++u) {
            const int j = j0 + u * SP_THREADS;
            if (j >= N || j == i || __ldcg(s.dead + jj[u])) continue;
            const double q = acc[u];
            if (!(q < worst)) continue;
            int r = D - 1;
            while (r > 0 && list[(r - 1) * SP_THREADS + tid] > q) {
                list[r * SP_THREADS + tid] = list[(r - 1) * SP_THREADS + tid];
                --r;
            }
            list[r * SP_THREADS + tid] = q;
            worst = list[(D - 1) * SP_THREADS + tid];
        }
    }
    int ptr = 0;
    double head = list[tid];
    double sum = 0.0, last = 0.0;
    for (int r = 0; r < D; ++r) {
        double v = head;
        int w = tid;
        block_min_pair(v, w, red_v, red_w);
        if (w == tid) head = (++ptr < D) ? list[ptr * SP_THREADS + tid] : INFINITY;
        sum = __dadd_rn(sum, __dsqrt_rn(v));
        last = v;
    }
    if (tid == 0) {
        s.dens[i] = sum;
        s.thr2[i] = last;
    }
}

// (dens, index) minimum over this block's slice of live rows -> bval / bidx[blockIdx.x]
__device__ void slice_min(const SpState& s, double* red_v, int* red_w)
{
    double v = INFINITY;
    int w = INT_MAX;
    for (int i = blockIdx.x * SP_THREADS + threadIdx.x; i < s.N; i += gridDim.x * SP_THREADS) {
        if (__ldcg(s.dead + i)) continue;
        const double d = __ldcg(s.dens + i);
        if (pair_less(d, i, v, w)) { v = d; w = i; }
    }
    block_min_pair(v, w, red_v, red_w);
    if (threadIdx.x == 0) {
        s.bval[blockIdx.x] = v;
        s.bidx[blockIdx.x] = w;
    }
}

__global__ void __launch_bounds__(SP_THREADS) lb_sparsify_kernel(SpState s)
{
    extern __shared__ double list[]; // D x SP_THREADS
    __shared__ double sh_x[LB_MAX_D];
    __shared__ double red_v[33];
    __shared__ int red_w[33];
    cg::grid_group grid = cg::this_grid();
    const int G = gridDim.x, b = blockIdx.x, tid = threadIdx.x;

    for (int i = b; i < s.N; i += G) score_row(s, i, list, sh_x, red_v, red_w);
    grid.sync();
    slice_min(s, red_v, red_w);
    grid.sync();

    for (int t = 0; t < s.n_remove; ++t) {
        // S1: the removed point, then the rows whose D nearest it was among
        double v = INFINITY;
        int w = INT_MAX;
        for (int g = tid; g < G; g += SP_THREADS) {
            const double gv = __ldcg(s.bval + g);
            const int gw = __ldcg(s.bidx + g);
            if (pair_less(gv, gw, v, w)) { v = gv; w = gw; }
        }
        block_min_pair(v, w, red_v, red_w);
        const int k = w;
        if (b == 0 && tid == 0) {
            s.rem_idx[t] = k;
            s.rem_dens[t] = v;
            s.dead[k] = 1;
            s.count[(t + 1) & 1] = 0; // last read in S2 of removal t - 1
        }
        if (t + 1 == s.n_remove) break;
        if (tid < s.D) sh_x[tid] = __ldg(s.X + (size_t)tid * s.N + k);
        __syncthreads();
        int* cnt = s.count + (t & 1);
        for (int i = b * SP_THREADS + tid; i < s.N; i += G * SP_THREADS) {
            if (i == k || __ldcg(s.dead + i)) continue;
            if (sq_dist(s.X, s.N, s.D, sh_x, i) <= __ldcg(s.thr2 + i)) s.work[atomicAdd(cnt, 1)] = i;
        }
        grid.sync();
        // S2: re-score the affected rows over the live points
        const int nw = __ldcg(cnt);
        for (int p = b; p < nw; p += G) score_row(s, __ldcg(s.work + p), list, sh_x, red_v, red_w);
        grid.sync();
        // S3
        slice_min(s, red_v, red_w);
        grid.sync();
    }
}

LbOncePerDevice g_smem_attr;

size_t align256(size_t b) { return (b + 255) / 256 * 256; }

} // namespace

extern "C" int lb_sparsify(lb_gp* h, int64_t N, int D, const double* X, int64_t max_points, int64_t* keep_idx,
    int64_t* removed_idx, double* removed_density)
{
    if (!h || N < 1 || N > INT_MAX || D < 1 || D > LB_MAX_D || max_points < D || !X || !keep_idx) return LB_ERR_ARG;
    if (N <= max_points) {
        for (int64_t i = 0; i < N; ++i) keep_idx[i] = i;
        return LB_OK;
    }
    LB_DEVICE(h);
    const int n = (int)N, R = (int)(N - max_points);
    const size_t smem = sizeof(double) * (size_t)D * SP_THREADS;
    if (g_smem_attr.need())
        LB_CUDA(cudaFuncSetAttribute(lb_sparsify_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
            (int)(sizeof(double) * LB_MAX_D * SP_THREADS)));
    int dev = 0, sms = 0, coop = 0, per_sm = 0;
    LB_CUDA(cudaGetDevice(&dev));
    LB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    LB_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
    if (!coop) return LB_ERR_UNSUPPORTED;
    LB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, lb_sparsify_kernel, SP_THREADS, smem));
    if (per_sm < 1) return LB_ERR_UNSUPPORTED;
    const int G = sms * std::min(per_sm, SP_MAX_BLOCKS_PER_SM);

    // scratch: X | dens | thr2 | rem_dens | bval | dead, count | work | rem_idx | bidx
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += align256(bytes); return o; };
    const size_t oX = take(sizeof(double) * (size_t)D * n), oDens = take(sizeof(double) * n), oThr = take(sizeof(double) * n),
                 oRemD = take(sizeof(double) * R), oBval = take(sizeof(double) * G), oDead = take(sizeof(int) * ((size_t)n + 2)),
                 oWork = take(sizeof(int) * n), oRemI = take(sizeof(int) * R), oBidx = take(sizeof(int) * G);
    int rc = lb_ensure_scratch(h, off);
    if (rc) return rc;
    char* base = reinterpret_cast<char*>(h->dScratch);

    std::vector<double> soa((size_t)D * n);
    for (int i = 0; i < n; ++i)
        for (int d = 0; d < D; ++d) soa[(size_t)d * n + i] = X[(size_t)i * D + d];
    LB_CUDA(cudaMemcpyAsync(base + oX, soa.data(), sizeof(double) * soa.size(), cudaMemcpyHostToDevice, h->stream));
    LB_CUDA(cudaMemsetAsync(base + oDead, 0, sizeof(int) * ((size_t)n + 2), h->stream));

    SpState s;
    s.X = reinterpret_cast<const double*>(base + oX);
    s.N = n; s.D = D; s.n_remove = R;
    s.dens = reinterpret_cast<double*>(base + oDens);
    s.thr2 = reinterpret_cast<double*>(base + oThr);
    s.dead = reinterpret_cast<int*>(base + oDead);
    s.count = s.dead + n;
    s.work = reinterpret_cast<int*>(base + oWork);
    s.bval = reinterpret_cast<double*>(base + oBval);
    s.bidx = reinterpret_cast<int*>(base + oBidx);
    s.rem_idx = reinterpret_cast<int*>(base + oRemI);
    s.rem_dens = reinterpret_cast<double*>(base + oRemD);
    void* args[] = {&s};
    LB_CUDA(cudaLaunchCooperativeKernel((const void*)lb_sparsify_kernel, dim3(G), dim3(SP_THREADS), args, smem, h->stream));
    h->launches++;

    std::vector<int> ridx(R);
    std::vector<double> rdens(R);
    LB_CUDA(cudaMemcpyAsync(ridx.data(), s.rem_idx, sizeof(int) * R, cudaMemcpyDeviceToHost, h->stream));
    if (removed_density)
        LB_CUDA(cudaMemcpyAsync(rdens.data(), s.rem_dens, sizeof(double) * R, cudaMemcpyDeviceToHost, h->stream));
    LB_CUDA(cudaStreamSynchronize(h->stream));
    std::vector<char> gone(n, 0);
    for (int t = 0; t < R; ++t) {
        if (ridx[t] < 0 || ridx[t] >= n || gone[ridx[t]]) return LB_ERR_STATE;
        gone[ridx[t]] = 1;
        if (removed_idx) removed_idx[t] = ridx[t];
        if (removed_density) removed_density[t] = rdens[t];
    }
    for (int i = 0, m = 0; i < n; ++i)
        if (!gone[i]) keep_idx[m++] = i;
    return LB_OK;
}
