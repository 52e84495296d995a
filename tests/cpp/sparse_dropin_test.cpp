// tests/cpp/sparse_dropin_test.cpp — limbo_b200::model::SparsifiedGP next to the reference's own limbo::model::SparsifiedGP
// (/root/reference/src/limbo/model/sparsified_gp.hpp), alone and as the GPClass of the reference's limbo::model::MultiGP,
// on the reference's test configuration (src/tests/test_gp.cpp:760-800: D = 1, 100 samples, max_points = 33, SquaredExpARD,
// KernelLFOpt<Rprop>).  Kept samples must be identical; predictions agree to the fp64 bar.  Needs a GPU to run.
// (Eigen is the stand-in from oracle/ref_sparse + oracle/ref_shim because the image has no Eigen.)
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <limbo/kernel/matern_five_halves.hpp>
#include <limbo/kernel/squared_exp_ard.hpp>
#include <limbo/mean/constant.hpp>
#include <limbo/mean/data.hpp>
#include <limbo/model/gp.hpp>
#include <limbo/model/gp/kernel_lf_opt.hpp>
#include <limbo/model/gp/no_lf_opt.hpp>
#include <limbo/model/sparsified_gp.hpp>
#include <limbo/model/multi_gp.hpp>
#include <limbo/opt/rprop.hpp>

#include <limbo_b200/model/sparsified_gp.hpp>

using namespace limbo;

struct Params {
    struct kernel : public defaults::kernel {};
    struct kernel_squared_exp_ard : public defaults::kernel_squared_exp_ard {};
    struct kernel_maternfivehalves : public defaults::kernel_maternfivehalves {};
    struct mean_constant : public defaults::mean_constant {};
    struct opt_rprop {
        BO_PARAM(int, iterations, 20);
        BO_PARAM(double, eps_stop, 0.0);
    };
    struct model_sparse_gp {
        BO_PARAM(int, max_points, 100 / 3);
    };
};

static double u01(unsigned long long& s)
{ // splitmix64, as limbo_b200/synth.py
    s += 0x9E3779B97F4A7C15ULL;
    unsigned long long z = s;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    z ^= z >> 31;
    return (double)(z >> 11) * (1.0 / 9007199254740992.0);
}

static Eigen::VectorXd vec(std::initializer_list<double> v)
{
    Eigen::VectorXd x((Eigen::Index)v.size());
    Eigen::Index i = 0;
    for (double a : v) x(i++) = a;
    return x;
}

static bool same_samples(const std::vector<Eigen::VectorXd>& a, const std::vector<Eigen::VectorXd>& b)
{
    if (a.size() != b.size()) return false;
    for (size_t i = 0; i < a.size(); ++i)
        for (Eigen::Index d = 0; d < a[i].size(); ++d)
            if (a[i](d) != b[i](d)) return false;
    return true;
}

static double absdiff(double a, double b) { return std::abs(a - b); }
static double absdiff(const Eigen::VectorXd& a, const Eigen::VectorXd& b)
{
    double e = 0;
    for (Eigen::Index i = 0; i < a.size(); ++i) e = std::max(e, std::abs(a(i) - b(i)));
    return e;
}

template <typename A, typename B>
static double max_mu_diff(const A& ra, const B& rb, const std::vector<Eigen::VectorXd>& Q)
{
    double e = 0;
    for (const auto& q : Q) {
        auto a = ra.query(q);
        auto b = rb.query(q);
        e = std::max(e, absdiff(std::get<0>(a), std::get<0>(b)));
        e = std::max(e, absdiff(std::get<1>(a), std::get<1>(b)));
    }
    return e;
}

int main()
{
    int bad = 0;
    unsigned long long seed = 7;
    std::vector<Eigen::VectorXd> X, Y, Q;
    for (int i = 0; i < 110; ++i) {
        const double x = 10 * u01(seed);
        X.push_back(vec({x}));
        Y.push_back(vec({std::cos(x), std::sin(0.5 * x)}));
    }
    for (int i = 0; i < 20; ++i) Q.push_back(vec({10 * u01(seed)}));
    std::vector<Eigen::VectorXd> X0(X.begin(), X.begin() + 100), Y1;
    for (int i = 0; i < 110; ++i) Y1.push_back(vec({Y[i](0)}));
    std::vector<Eigen::VectorXd> Y10(Y1.begin(), Y1.begin() + 100), Y0(Y.begin(), Y.begin() + 100);

    // SparsifiedGP: compute, Rprop, then add_sample past the cap
    using KF = kernel::SquaredExpARD<Params>;
    using HP = model::gp::KernelLFOpt<Params, opt::Rprop<Params>>;
    model::SparsifiedGP<Params, KF, mean::Constant<Params>, HP> ref(1, 1);
    limbo_b200::model::SparsifiedGP<Params, KF, mean::Constant<Params>, HP> gpu(1, 1);
    ref.compute(X0, Y10);
    gpu.compute(X0, Y10);
    const bool kept = same_samples(ref.samples(), gpu.samples()) && gpu.samples().size() == 33;
    const double e0 = max_mu_diff(ref, gpu, Q);
    ref.optimize_hyperparams();
    gpu.optimize_hyperparams();
    const double ehp = absdiff(ref.kernel_function().h_params(), gpu.kernel_function().h_params());
    for (int i = 100; i < 110; ++i) {
        ref.add_sample(X[i], Y1[i]);
        gpu.add_sample(X[i], Y1[i]);
    }
    const bool kept_add = same_samples(ref.samples(), gpu.samples());
    const double e1 = max_mu_diff(ref, gpu, Q);
    std::printf("SparsifiedGP: kept %d |dmu,ds2| %.3g  Rprop |dhp| %.3g  add_sample kept %d |dmu,ds2| %.3g\n", kept, e0, ehp, kept_add, e1);
    bad += !(kept && e0 <= 1e-9 && ehp <= 1e-7 && kept_add && e1 <= 1e-7);

    // MultiGP<Params, SparsifiedGP, ...>: two outputs over the same kept samples
    using KM = kernel::MaternFiveHalves<Params>;
    model::MultiGP<Params, model::SparsifiedGP, KM, mean::Data<Params>> mref;
    model::MultiGP<Params, limbo_b200::model::SparsifiedGP, KM, mean::Data<Params>> mgpu;
    mref.compute(X0, Y0);
    mgpu.compute(X0, Y0);
    const bool mkept = same_samples(mref.gp_models()[0].samples(), mgpu.gp_models()[0].samples())
        && same_samples(mref.gp_models()[1].samples(), mgpu.gp_models()[1].samples());
    for (int i = 100; i < 105; ++i) {
        mref.add_sample(X[i], Y[i]);
        mgpu.add_sample(X[i], Y[i]);
    }
    const bool mkept_add = same_samples(mref.gp_models()[0].samples(), mgpu.gp_models()[0].samples());
    const double em = max_mu_diff(mref, mgpu, Q);
    std::printf("MultiGP<SparsifiedGP>: kept %d  add_sample kept %d |dmu,ds2| %.3g\n", mkept, mkept_add, em);
    bad += !(mkept && mkept_add && em <= 1e-9);
    std::printf(bad ? "SPARSE DROPIN FAIL\n" : "SPARSE DROPIN OK\n");
    return bad;
}
