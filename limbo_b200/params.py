"""Parameter plumbing mirroring limbo's ``Params::section::name()`` statics
(src/limbo/tools/macros.hpp:53-123): a Params class holds nested classes, one
per section; anything missing falls back to the reference default."""
from __future__ import annotations


class defaults:
    class kernel:  # kernel/kernel.hpp:54-59
        noise = 0.01
        optimize_noise = False

    class kernel_squared_exp_ard:  # kernel/squared_exp_ard.hpp:53-59
        k = 0
        sigma_sq = 1.0

    class kernel_maternfivehalves:  # kernel/matern_five_halves.hpp:53-59
        sigma_sq = 1.0
        l = 1.0

    class kernel_maternthreehalves:  # kernel/matern_three_halves.hpp:53-59
        sigma_sq = 1.0
        l = 1.0

    class kernel_exp:  # kernel/exp.hpp:53-59
        sigma_sq = 1.0
        l = 1.0

    class mean_constant:  # mean/constant.hpp:54-57
        constant = 1.0

    class acqui_ucb:  # acqui/ucb.hpp:55-58
        alpha = 0.5

    class acqui_gpucb:  # acqui/gp_ucb.hpp:55-58
        delta = 0.1

    class acqui_ei:  # acqui/ei.hpp:57-60
        jitter = 0.0

    class opt_rprop:  # opt/rprop.hpp:58-65
        iterations = 300
        eps_stop = 0.0

    class opt_parallelrepeater:  # opt/parallel_repeater.hpp:59-66
        repeats = 10
        epsilon = 1e-2

    class model_sparse_gp:  # model/sparsified_gp.hpp:56-59
        max_points = 200

    class bayes_opt_boptimizer:  # bayes_opt/boptimizer.hpp:68-72
        hp_period = -1


class Params:
    """Empty parameter set = all reference defaults; subclass and add sections to override."""


def get(params, section: str, name: str):
    sec = getattr(params, section, None) if params is not None else None
    if sec is not None and hasattr(sec, name):
        return getattr(sec, name)
    return getattr(getattr(defaults, section), name)
