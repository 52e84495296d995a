// include/limbo_b200/model/sparsified_gp.hpp — drop-in for limbo::model::SparsifiedGP (src/limbo/model/sparsified_gp.hpp:77-183)
// over limbo_b200::model::GP.  Same template signature, so it is also the GPClass argument of the reference's
// limbo::model::MultiGP<Params, GPClass, Kernel, Mean>.  The density-based selection runs on the device (lb_sparsify, one
// launch); the fit of the kept samples is limbo_b200::model::GP::compute.  Reads Params::model_sparse_gp::max_points()
// (limbo::defaults::model_sparse_gp has the reference's default, 200).
#ifndef LIMBO_B200_MODEL_SPARSIFIED_GP_HPP
#define LIMBO_B200_MODEL_SPARSIFIED_GP_HPP

#include <limbo_b200/model/gp.hpp>

namespace limbo_b200 {
    namespace model {
        template <typename Params, typename KernelFunction, typename MeanFunction, typename HyperParamsOptimizer>
        class SparsifiedGP : public GP<Params, KernelFunction, MeanFunction, HyperParamsOptimizer> {
        public:
            using base_gp_t = GP<Params, KernelFunction, MeanFunction, HyperParamsOptimizer>;

            SparsifiedGP() : base_gp_t() {}
            SparsifiedGP(int dim_in, int dim_out) : base_gp_t(dim_in, dim_out) {}

            // sparsified_gp.hpp:84-101.  Throws std::runtime_error when max_points() is smaller than the input dimension
            // (the reference's partial_sort would read past its row).
            void compute(const std::vector<Eigen::VectorXd>& samples, const std::vector<Eigen::VectorXd>& observations,
                bool compute_kernel = true)
            {
                const long cap = Params::model_sparse_gp::max_points();
                if ((long)samples.size() <= cap) {
                    base_gp_t::compute(samples, observations, compute_kernel);
                    return;
                }
                const long N = (long)samples.size();
                const int D = (int)samples.front().size();
                std::vector<double> x((size_t)N * D);
                for (long i = 0; i < N; ++i)
                    for (int d = 0; d < D; ++d) x[(size_t)i * D + d] = samples[i](d);
                std::vector<int64_t> keep((size_t)cap);
                lb_check(lb_sparsify(this->_h, N, D, x.data(), cap, keep.data(), nullptr, nullptr), "lb_sparsify");
                std::vector<Eigen::VectorXd> samp, obs;
                for (int64_t k : keep) {
                    samp.push_back(samples[(size_t)k]);
                    obs.push_back(observations[(size_t)k]);
                }
                base_gp_t::compute(samp, obs, compute_kernel);
            }

            // sparsified_gp.hpp:105-119.  Past the cap the reference appends the sample, then re-sparsifies the current
            // samples plus the new one and refits from scratch; only the refit is observable, so the append is skipped.
            void add_sample(const Eigen::VectorXd& sample, const Eigen::VectorXd& observation)
            {
                if ((long)this->_samples.size() + 1 <= (long)Params::model_sparse_gp::max_points()) {
                    base_gp_t::add_sample(sample, observation);
                    return;
                }
                std::vector<Eigen::VectorXd> samp = this->_samples, obs;
                samp.push_back(sample);
                for (long i = 0; i < (long)this->_observations.rows(); ++i) {
                    Eigen::VectorXd o(this->_observations.cols());
                    for (Eigen::Index p = 0; p < this->_observations.cols(); ++p) o(p) = this->_observations(i, p);
                    obs.push_back(o);
                }
                obs.push_back(observation);
                compute(samp, obs, true);
            }
        };
    } // namespace model
} // namespace limbo_b200

#endif
