"""model::MultiGP (src/limbo/model/multi_gp.hpp:60-397): dim_out independent single-output GPs over the same samples.

Structure as in the reference: the inner GPs are built with mean::NullFunction and no hyper-parameter optimiser
(multi_gp.hpp:63), ONE mean function of width dim_out lives at the MultiGP level, is subtracted from the observations
before they are split per output (multi_gp.hpp:112-118) and added back to the predictions (multi_gp.hpp:183-203), so
coupled means (mean::FunctionARD) and their h-params behave like the reference's.  The reference fans the per-output
work over tools::par; here every inner GP is its own device handle (own stream), optionally on its own GPU."""
from __future__ import annotations

import numpy as np

from .. import kernel as _kernel
from .. import mean as _mean
from .gp import GP


class MultiGP:
    def __init__(self, dim_in: int = -1, dim_out: int = -1, params=None, kernel=_kernel.MaternFiveHalves, mean=_mean.Data,
                 hp_opt=None, device: int = 0, devices=None, gp=GP):
        # gp: the per-output model class, the reference's template-template argument (multi_gp.hpp:59), e.g. SparsifiedGP
        self._gp_cls = gp
        self._params = params
        self._kernel_cls, self._mean_cls = kernel, mean
        self._dim_in, self._dim_out = dim_in, dim_out
        self._devices = list(devices) if devices else [device]
        self._mean_function = mean(params, dim_out if dim_out > 0 else 1)
        self._gp_models: list[GP] = []
        self._observations = np.zeros((0, max(dim_out, 1)))
        self._mean_observation = np.zeros(max(dim_out, 1))
        if hp_opt is None:
            from .hp_opt import NoLFOpt
            hp_opt = NoLFOpt(params)
        self._hp_optimize = hp_opt
        if dim_out > 0:  # multi_gp.hpp:71-78
            self._gp_models = [self._make_gp(i) for i in range(dim_out)]

    def _make_gp(self, i: int) -> GP:
        return self._gp_cls(self._dim_in if self._dim_in > 0 else -1, 1, params=self._params, kernel=self._kernel_cls, mean=_mean.NullFunction,
                  device=self._devices[i % len(self._devices)])

    def _update_mean_observation(self) -> None:
        self._mean_observation = self._observations.mean(axis=0) if len(self._observations) else np.zeros(max(self._dim_out, 1))

    # ---- multi_gp.hpp:81-127 ----
    def compute(self, samples, observations, compute_kernel: bool = True) -> None:
        assert len(samples) != 0 and len(observations) != 0 and len(samples) == len(observations)
        X = np.array(samples, dtype=np.float64, copy=True)
        Y = np.array(observations, dtype=np.float64, copy=True)
        if X.ndim == 1:
            X = X[:, None]
        if Y.ndim == 1:
            Y = Y[:, None]
        self._dim_in = X.shape[1]
        if self._dim_out != Y.shape[1]:
            self._dim_out = Y.shape[1]
            self._mean_function = self._mean_cls(self._params, self._dim_out)
        if len(self._gp_models) != self._dim_out:
            self._gp_models = [self._make_gp(i) for i in range(self._dim_out)]
        self._observations = Y
        self._update_mean_observation()
        M = np.asarray(self._mean_function.batch(X, self), dtype=np.float64).reshape(len(X), self._dim_out)
        obs = Y - M
        for i, gp in enumerate(self._gp_models):
            gp.compute(X, obs[:, i:i + 1], compute_kernel)

    def optimize_hyperparams(self) -> None:  # multi_gp.hpp:130-133
        self._hp_optimize(self)

    def mean_function(self):
        return self._mean_function

    # ---- multi_gp.hpp:139-176 ----
    def add_sample(self, sample, observation) -> None:
        sample = np.atleast_1d(np.asarray(sample, dtype=np.float64))
        observation = np.atleast_1d(np.asarray(observation, dtype=np.float64))
        if not self._gp_models:
            self._dim_in = sample.size
            if self._dim_out != observation.size:
                self._dim_out = observation.size
                self._mean_function = self._mean_cls(self._params, self._dim_out)
            self._gp_models = [self._make_gp(i) for i in range(self._dim_out)]
            self._observations = np.zeros((0, self._dim_out))
        else:
            assert sample.size == self._dim_in
            assert observation.size == self._dim_out
        self._observations = np.vstack([self._observations.reshape(-1, self._dim_out), observation[None, :]])
        self._update_mean_observation()
        mean_vector = np.asarray(self._mean_function(sample, self), dtype=np.float64)
        assert mean_vector.size == self._dim_out
        for i, gp in enumerate(self._gp_models):
            gp.add_sample(sample, np.array([observation[i] - mean_vector[i]]))

    # ---- multi_gp.hpp:183-232 ----
    def query(self, v):
        v = np.asarray(v, dtype=np.float64)
        mean_vector = np.asarray(self._mean_function(v, self), dtype=np.float64)
        mu, sigma = np.empty(self._dim_out), np.empty(self._dim_out)
        for i, gp in enumerate(self._gp_models):
            m, s = gp.query(v)
            mu[i] = m[0] + mean_vector[i]
            sigma[i] = s
        return mu, sigma

    def query_batch(self, Xq):
        """mu (M x dim_out) and sigma^2 (M x dim_out): one batched device pass per output."""
        Xq = np.ascontiguousarray(np.atleast_2d(Xq), dtype=np.float64)
        res = [gp.query_batch(Xq) for gp in self._gp_models]
        M = np.asarray(self._mean_function.batch(Xq, self), dtype=np.float64).reshape(len(Xq), self._dim_out)
        return np.concatenate([r[0] for r in res], axis=1) + M, np.stack([r[1] for r in res], axis=1)

    def mu(self, v):
        return self.query(v)[0]

    def sigma(self, v):
        return np.array([gp.sigma(v) for gp in self._gp_models])

    def dim_in(self):
        assert self._dim_in != -1
        return self._dim_in

    def dim_out(self):
        assert self._dim_out != -1
        return self._dim_out

    def nb_samples(self):
        return len(self._observations)

    # ---- multi_gp.hpp:253-266 ----
    def recompute(self, update_obs_mean: bool = True, update_full_kernel: bool = True) -> None:
        if not self._gp_models:
            return
        if update_obs_mean:  # "if the mean is updated, we need to fully re-compute"
            return self.compute(np.stack(self._gp_models[0].samples()), self._observations, update_full_kernel)
        for gp in self._gp_models:
            gp.recompute(False, update_full_kernel)

    def samples(self):
        assert self._gp_models
        return self._gp_models[0].samples()

    def observations(self):
        return [self._observations[i] for i in range(len(self._observations))]

    def observations_matrix(self) -> np.ndarray:
        assert self._dim_out > 0
        return self._observations

    def mean_observation(self) -> np.ndarray:
        assert self._dim_out > 0
        return self._mean_observation if len(self._observations) else np.zeros(self._dim_out)

    def gp_models(self):
        return self._gp_models

    # ---- multi_gp.hpp:314-390 ----
    def save(self, archive) -> None:
        from ..serialize import TextArchive
        if isinstance(archive, str):
            archive = TextArchive(archive)
        archive.save(np.array([float(self._dim_in), float(self._dim_out)]), "dims")
        archive.save(self._observations, "observations")
        if self._mean_function.h_params_size() > 0:
            archive.save(self._mean_function.h_params(), "mean_params")
        for i, gp in enumerate(self._gp_models):
            gp.save(type(archive)(archive.directory() + "/gp_" + str(i)))

    def load(self, archive, recompute: bool = True) -> None:
        from ..serialize import TextArchive
        if isinstance(archive, str):
            archive = TextArchive(archive)
        self._observations = archive.load_matrix("observations")
        dims = archive.load_vector("dims")
        self._dim_in, self._dim_out = int(dims[0]), int(dims[1])
        self._observations = self._observations.reshape(-1, self._dim_out)
        self._update_mean_observation()
        self._mean_function = self._mean_cls(self._params, self._dim_out)
        if self._mean_function.h_params_size() > 0:
            hp = archive.load_vector("mean_params")
            assert hp.size == self._mean_function.h_params_size()
            self._mean_function.set_h_params(hp)
        self._gp_models = [self._make_gp(i) for i in range(self._dim_out)]
        for i, gp in enumerate(self._gp_models):
            gp.load(type(archive)(archive.directory() + "/gp_" + str(i)), recompute=False)
        if recompute:
            self.recompute(True, True)
