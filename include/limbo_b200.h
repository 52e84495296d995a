/* include/limbo_b200.h — C ABI of the B200-native GP compute backend for Limbo.
 *
 * The reference (resibots/limbo @ 43c67a6) has no FFI for this path: the seam
 * is the C++ "Model concept" implemented by limbo::model::GP
 * (src/limbo/model/gp.hpp:81-511).  This header is the boundary a drop-in
 * model type binds to (include/limbo_b200/model/gp.hpp does exactly that, and
 * INTEGRATION.md shows the maintainer-side glue).  Each entry point names the
 * reference member it replaces.
 *
 * Conventions
 *   - all pointers are HOST pointers unless the function name ends in _dev;
 *   - matrices are column-major like Eigen::MatrixXd; sample/candidate arrays
 *     are row-major "one point per row" (the reference holds them as
 *     std::vector<Eigen::VectorXd>);
 *   - mean functions stay on the host (they are arbitrary user functors,
 *     src/limbo/mean/mean.hpp:60-77): callers pass obs_mean = Y - M
 *     (gp.hpp:547) and add mean(v) to the returned mu (gp.hpp:615);
 *   - every function returns 0 on success; > 0 = 1-based index of the first
 *     non-positive Cholesky pivot (LAPACK-style info; the reference never
 *     checks Eigen's info(), gp.hpp:565); < 0 = LB_ERR_*;
 *   - lb_query / lb_acq_argmax on one handle may be called from several host
 *     threads (the reference's query() is const and called concurrently from
 *     TBB workers, opt/parallel_repeater.hpp:103); mutating calls need
 *     exclusive access to the handle.
 *   - there is no CPU fallback: without a CUDA device lb_create fails.
 */
#ifndef LIMBO_B200_H
#define LIMBO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct lb_gp lb_gp;

#define LB_OK 0
#define LB_ERR_ARG (-1)
#define LB_ERR_CUDA (-2)
#define LB_ERR_STATE (-3)
#define LB_ERR_ALLOC (-4)
#define LB_ERR_UNSUPPORTED (-5)
#define LB_ERR_TIMEOUT (-6)

/* kernel ids (the functors under src/limbo/kernel/) */
#define LB_KERNEL_SQUARED_EXP_ARD 0 /* kernel/squared_exp_ard.hpp   h-params [log l_1..log l_D, (A(:,0) .. A(:,k-1): D each, k <= 4), log sigma_f];
                                       k = Params::kernel_squared_exp_ard::k() is inferred from n_hparams = D + D k + 1 */
#define LB_KERNEL_MATERN_FIVE_HALVES 1 /* kernel/matern_five_halves.hpp      h-params [log l, log sigma_f] */
#define LB_KERNEL_MATERN_THREE_HALVES 2 /* kernel/matern_three_halves.hpp */
#define LB_KERNEL_EXP 3 /* kernel/exp.hpp */

/* acquisition ids */
#define LB_ACQ_UCB 0 /* acqui/ucb.hpp:83-90 and acqui/gp_ucb.hpp:96-103; params[0] = alpha (resp. beta) */
#define LB_ACQ_EI 1  /* acqui/ei.hpp:85-116; params[0] = f_max, params[1] = jitter */

/* lb_get selectors */
#define LB_GET_K 0     /* _kernel     gp.hpp:553-562 (N x N, both triangles) */
#define LB_GET_L 1     /* _matrixL    gp.hpp:565     (N x N, zero upper part) */
#define LB_GET_ALPHA 2 /* _alpha      gp.hpp:605-611 (N x P) */
#define LB_GET_KINV 3  /* _inv_kernel gp.hpp:254-264 (N x N) */

/* precision modes */
#define LB_PREC_FP64 0
/* fit / likelihood in fp64; lb_query and lb_acq_argmax compute sigma^2 on the tf32 tensor cores (tcgen05, fp32
 * accumulation) from an fp64-inverted factor; mu stays fp64.  |d sigma^2| = a few 1e-3 k(v,v), growing with cond(K)
 * (measured maxima in tests/test_gpu_tf32.py) */
#define LB_PREC_TF32 1
/* same path with fp16 operands (same 11-bit significand as tf32, half the operand bytes, twice the tensor rate);
 * K* is scaled by 1/sigma_f^2 and L^-1 by a power of two so that both stay inside the fp16 range */
#define LB_PREC_FP16 2
/* fp16 split operands: every operand is hi + 2^-11 lo (two fp16 planes, 22 significant bits), three tensor-core products per
 * k-step, hi x hi and the cross terms in separate fp32 accumulators, combined and squared in fp64.  About 3x the scoring time of
 * LB_PREC_FP16; |d sigma^2| <= 2e-5 k(v,v) up to N = 4096 and <= 1e-4 at N = 16384, cond(K) ~ 1.6e6 (the fp32 accumulation of the
 * tensor core is the floor there; tests/test_gpu_tf32.py, tests/test_gpu_config4.py), against 2-4e-3 for the one-plane modes */
#define LB_PREC_FP16X3 3

/* Lifetime.  Replaces GP(int dim_in, int dim_out) / ~GP / the copy constructor
 * KernelLFOptimization relies on (model/gp/kernel_lf_opt.hpp:79). */
int lb_create(lb_gp** out, int device, int precision);
int lb_destroy(lb_gp* h);
int lb_clone(const lb_gp* h, lb_gp** out);

/* Run all work of this handle on an existing CUDA stream (cudaStream_t cast
 * to void*); NULL restores the handle's own stream. */
int lb_set_stream(lb_gp* h, void* cuda_stream);
int lb_sync(lb_gp* h);
/* number of kernels launched by this handle so far */
long long lb_launch_count(const lb_gp* h);

/* GP::compute data part (gp.hpp:88-116): N samples of dimension D (row-major
 * N x D) and obs_mean = observations - mean (column-major N x P). */
int lb_set_data(lb_gp* h, int64_t N, int D, int P, const double* X_rowmajor, const double* obs_mean_colmajor);
int lb_set_data_dev(lb_gp* h, int64_t N, int D, int P, const double* dX_rowmajor, const double* dObsMean_colmajor);

/* Kernel functor state: BaseKernel::set_h_params (kernel/kernel.hpp:116-123).
 * log_hparams are the kernel's own log-space parameters (without the noise
 * entry); noise is the signal noise itself (kernel.hpp:126). */
int lb_set_kernel(lb_gp* h, int kernel_id, const double* log_hparams, int n_hparams, double noise);

/* GP::_compute_full_kernel (gp.hpp:550-571): K -> L -> alpha. */
int lb_fit(lb_gp* h);
/* GP::recompute(update_obs_mean, update_full_kernel=false) (gp.hpp:241-252):
 * new obs_mean, same factor, re-solve alpha. */
int lb_refit_alpha(lb_gp* h, const double* obs_mean_colmajor);
/* GP::add_sample / _compute_incremental_kernel (gp.hpp:126-152, 573-603):
 * x is the new sample (D), obs_mean_all the refreshed (N+1) x P obs_mean. */
int lb_append(lb_gp* h, const double* x, const double* obs_mean_all_colmajor);

/* GP::load(archive, recompute = false) (gp.hpp:505-509): adopt a stored factor (N x N column-major, lower) and alpha
 * (N x P) for the data / kernel already set, instead of refactorising. */
int lb_load_factor(lb_gp* h, const double* L_colmajor, const double* alpha_colmajor);

/* Batched GP::query (gp.hpp:159-167) for M candidates (row-major M x D):
 * mu_minus_mean is M x P row-major (k^T alpha, WITHOUT mean(v));
 * sigma2 is M (clamped as gp.hpp:623, + noise as gp.hpp:166).
 * With N == 0 returns the prior (gp.hpp:161-163). */
int lb_query(const lb_gp* h, int64_t M, const double* Xq_rowmajor, double* mu_minus_mean, double* sigma2);
int lb_query_dev(const lb_gp* h, int64_t M, const double* dXq_rowmajor, double* dMu_minus_mean, double* dSigma2);

/* Batched acquisition + argmax over M candidates with the FirstElem
 * aggregator (bayes_opt/bo_base.hpp:99-105).  mean_at_q: M values of the
 * first component of mean(v), or NULL to add mean_const to every mu.
 * acq_out (optional, M values) receives the acquisition values.  Ties resolve
 * to the lowest index, like the reference's sequential scan. */
int lb_acq_argmax(const lb_gp* h, int acq_id, const double* acq_params, int64_t M, const double* Xq_rowmajor,
    const double* mean_at_q, double mean_const, double* acq_out, double* best_val, int64_t* best_idx);
/* same, device pointers; d_best = {value, (double) index bit-copied as int64} */
int lb_acq_argmax_dev(const lb_gp* h, int acq_id, const double* acq_params, int64_t M, const double* dXq_rowmajor,
    const double* dMean_at_q, double mean_const, double* dAcq_out, double* dBest_val, int64_t* dBest_idx);

/* GP::compute_log_lik (gp.hpp:267-282) */
int lb_log_lik(lb_gp* h, double* out);
/* GP::compute_kernel_grad_log_lik (gp.hpp:285-311); grad has n_hparams
 * (+1 when optimize_noise, kernel.hpp:86-96) entries. */
int lb_kernel_grad_log_lik(lb_gp* h, int optimize_noise, double* grad);
/* GP::compute_inv_kernel (gp.hpp:254-264) */
int lb_compute_inv_kernel(lb_gp* h);

/* GP::compute_log_loo_cv (gp.hpp:339-351): leave-one-out log predictive probability from diag(K^-1) and alpha */
int lb_log_loo_cv(lb_gp* h, double* out);
/* GP::compute_kernel_grad_log_loo_cv (gp.hpp:353-399), the gradient KernelLooOpt (model/gp/kernel_loo_opt.hpp:57-97)
 * climbs; grad has n_hparams (+1 when optimize_noise) entries. */
int lb_kernel_grad_log_loo_cv(lb_gp* h, int optimize_noise, double* grad);
/* obs_mean^T K^-1 of GP::compute_mean_grad_log_lik (gp.hpp:313-330): out = K^-1 * obs_mean, N x P column-major; the
 * caller contracts it with its mean functor's gradient (mean/mean.hpp:72-76), which is host code. */
int lb_kinv_obs_mean(lb_gp* h, double* out_colmajor);

/* model::SparsifiedGP::_sparsify (model/sparsified_gp.hpp:126-183): greedy density-based selection of max_points of the N
 * samples (row-major N x D).  The density of a point is the sum of its D smallest Euclidean distances to the other
 * remaining points, added in ascending order; the point of smallest density is removed, the lowest index on a tie (the
 * reference's sequential scan), until max_points remain.  keep_idx receives the min(N, max_points) kept indices in
 * ascending order; removed_idx / removed_density (optional, NULL) the N - max_points removals in order and the density
 * at which each point went.  N <= max_points returns the identity and launches nothing.  LB_ERR_ARG for N < 1, D < 1,
 * D > 64 or max_points < D (the reference's partial_sort would then read past its row).  The handle's data, kernel,
 * factor and alpha are left as they are; its workspace is used, so the call needs exclusive access to the handle. */
int lb_sparsify(lb_gp* h, int64_t N, int D, const double* X_rowmajor, int64_t max_points,
    int64_t* keep_idx, int64_t* removed_idx, double* removed_density);

/* accessors matrixL(), alpha(), ... (gp.hpp:411-436): dst is column-major,
 * N x N (K, L, KINV) or N x P (ALPHA). */
int lb_get(lb_gp* h, int what, double* dst_colmajor);
int64_t lb_nb_samples(const lb_gp* h);

const char* lb_strerror(int code);
/* text of the last CUDA error seen by this library on the calling thread */
const char* lb_last_cuda_error(void);

#ifdef __cplusplus
}
#endif
#endif
