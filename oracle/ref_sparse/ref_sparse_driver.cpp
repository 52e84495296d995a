// oracle/ref_sparse/ref_sparse_driver.cpp — TEST INFRASTRUCTURE ONLY.
//
// Runs the REFERENCE'S OWN model::SparsifiedGP (src/limbo/model/sparsified_gp.hpp) and model::MultiGP over it
// (src/limbo/model/multi_gp.hpp) with mean::Data, on the Eigen stand-in (./Eigen, ../ref_shim/Eigen).  Used to write
// tests/golden/sparse/*.npz (tests/golden/make_golden_sparse.py) and to time the reference's selection
// (tools/sparsify_timing.py).  No reference source is copied: this file only instantiates its templates.
#include <limbo/kernel/matern_five_halves.hpp>
#include <limbo/kernel/squared_exp_ard.hpp>
#include <limbo/mean/data.hpp>
#include <limbo/model/gp.hpp>
#include <limbo/model/gp/kernel_lf_opt.hpp>
#include <limbo/model/gp/no_lf_opt.hpp>
#include <limbo/model/sparsified_gp.hpp>
#include <limbo/model/multi_gp.hpp>
#include <limbo/opt/rprop.hpp>
#include <chrono>
#include <tuple>

using namespace limbo;

struct SParams {
    struct kernel {
        BO_DYN_PARAM(double, noise);
        BO_PARAM(bool, optimize_noise, false);
    };
    struct kernel_squared_exp_ard : public defaults::kernel_squared_exp_ard {};
    struct kernel_maternfivehalves : public defaults::kernel_maternfivehalves {};
    struct opt_rprop {
        BO_DYN_PARAM(int, iterations);
        BO_PARAM(double, eps_stop, 0.0);
    };
    struct model_sparse_gp {
        BO_DYN_PARAM(int, max_points);
    };
};
BO_DECLARE_DYN_PARAM(double, SParams::kernel, noise);
BO_DECLARE_DYN_PARAM(int, SParams::opt_rprop, iterations);
BO_DECLARE_DYN_PARAM(int, SParams::model_sparse_gp, max_points);

namespace {

std::vector<Eigen::VectorXd> rows_of(const double* a, long n, int d)
{
    std::vector<Eigen::VectorXd> v;
    for (long i = 0; i < n; ++i) {
        Eigen::VectorXd x((Eigen::Index)d);
        for (int k = 0; k < d; ++k) x(k) = a[i * d + k];
        v.push_back(x);
    }
    return v;
}

// compute() on the first N0 samples, then add_sample() for the rest (N0 <= 0 or >= N: one compute over all N)
template <typename M>
double feed(M& m, const std::vector<Eigen::VectorXd>& s, const std::vector<Eigen::VectorXd>& o, long N0)
{
    const long N = (long)s.size();
    auto t0 = std::chrono::steady_clock::now();
    if (N0 > 0 && N0 < N) {
        m.compute(std::vector<Eigen::VectorXd>(s.begin(), s.begin() + N0), std::vector<Eigen::VectorXd>(o.begin(), o.begin() + N0));
        for (long i = N0; i < N; ++i) m.add_sample(s[i], o[i]);
    }
    else
        m.compute(s, o);
    return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
}

// The kept samples as original indices: a second SparsifiedGP fed the same samples with each sample's index as its
// observation (the selection depends on the samples only, and exact duplicates make matching by value ambiguous).
long kept_indices(long N, int D, const double* X, long N0, long* keep)
{
    using Idx_t = model::SparsifiedGP<SParams, kernel::MaternFiveHalves<SParams>, mean::Data<SParams>>;
    auto samples = rows_of(X, N, D);
    std::vector<Eigen::VectorXd> idx;
    for (long i = 0; i < N; ++i) {
        Eigen::VectorXd v(1);
        v(0) = (double)i;
        idx.push_back(v);
    }
    Idx_t g(D, 1);
    feed(g, samples, idx, N0);
    const long n = (long)g.samples().size();
    for (long i = 0; i < n; ++i) keep[i] = (long)g.observations()[i](0);
    return n;
}

template <typename Kernel>
int run(long N, int D, int P, const double* X, const double* Y, const double* hp, int nh, long N0, long M, const double* Xq,
    int rprop_iters, int multi, double* mu, double* s2, double* hp_out, double* seconds)
{
    auto samples = rows_of(X, N, D);
    auto obs = rows_of(Y, N, P);
    auto queries = rows_of(Xq, M, D);
    if (multi) {
        model::MultiGP<SParams, model::SparsifiedGP, Kernel, mean::Data<SParams>> gp(D, P);
        const double t = feed(gp, samples, obs, N0);
        if (seconds) *seconds = t;
        for (long q = 0; q < M; ++q) {
            Eigen::VectorXd m, s;
            std::tie(m, s) = gp.query(queries[q]);
            for (int p = 0; p < P; ++p) {
                mu[q * P + p] = m(p);
                s2[q * P + p] = s(p);
            }
        }
        return 0;
    }
    using GP_t = model::SparsifiedGP<SParams, Kernel, mean::Data<SParams>, model::gp::KernelLFOpt<SParams, opt::Rprop<SParams>>>;
    GP_t gp(D, P);
    if (hp) {
        Eigen::VectorXd h((Eigen::Index)nh);
        for (int i = 0; i < nh; ++i) h(i) = hp[i];
        gp.kernel_function().set_h_params(h);
    }
    const double t = feed(gp, samples, obs, N0);
    if (seconds) *seconds = t;
    if (rprop_iters > 0) {
        SParams::opt_rprop::set_iterations(rprop_iters);
        gp.optimize_hyperparams();
    }
    if (hp_out) {
        Eigen::VectorXd h = gp.kernel_function().h_params();
        for (Eigen::Index i = 0; i < h.size(); ++i) hp_out[i] = h(i);
    }
    for (long q = 0; q < M; ++q) {
        Eigen::VectorXd m;
        double s;
        std::tie(m, s) = gp.query(queries[q]);
        for (int p = 0; p < P; ++p) mu[q * P + p] = m(p);
        s2[q] = s;
    }
    return 0;
}

} // namespace

extern "C" {

// kernel_id: 0 SquaredExpARD, 1 MaternFiveHalves.  X: N x D, Y: N x P (row-major, raw observations: mean::Data is the
// reference's own).  keep (optional, max_points entries): kept original indices, their count in *n_keep.  mu: M x P;
// s2: M (multi = 0) or M x P (multi = 1, model::MultiGP<Params, model::SparsifiedGP, Kernel, mean::Data>).  seconds: wall
// time of the compute / add_sample sequence.  Y == NULL runs the index pass only.
int ref_sparse_gp_run(int kernel_id, long N, int D, int P, const double* X, const double* Y, double noise, const double* hp,
    int nh, long max_points, long N0, long M, const double* Xq, int rprop_iters, int multi, long* keep, long* n_keep, double* mu,
    double* s2, double* hp_out, double* seconds)
{
    SParams::kernel::set_noise(noise);
    SParams::model_sparse_gp::set_max_points((int)max_points);
    if (keep) {
        const long n = kept_indices(N, D, X, N0, keep);
        if (n_keep) *n_keep = n;
    }
    if (!Y) return 0;
    if (multi && (hp || rprop_iters > 0)) return 2;
    switch (kernel_id) {
    case 0: return run<kernel::SquaredExpARD<SParams>>(N, D, P, X, Y, hp, nh, N0, M, Xq, rprop_iters, multi, mu, s2, hp_out, seconds);
    case 1: return run<kernel::MaternFiveHalves<SParams>>(N, D, P, X, Y, hp, nh, N0, M, Xq, rprop_iters, multi, mu, s2, hp_out, seconds);
    default: return 1;
    }
}
}
