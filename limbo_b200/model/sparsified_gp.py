"""limbo_b200.model.SparsifiedGP — mirror of limbo::model::SparsifiedGP (src/limbo/model/sparsified_gp.hpp:77-183).

A GP that keeps at most Params::model_sparse_gp::max_points samples: past the cap it drops, one at a time, the sample of
smallest density (the sum of its D smallest distances to the other remaining samples, D the input dimension) and fits
the GP on what remains.  The selection runs on the device (lb_sparsify, one launch); the fit is GP.compute on the kept
samples and observations, so mean::Data averages the kept observations only."""
from __future__ import annotations

import ctypes as C

import numpy as np

from .. import _lib
from .. import kernel as _kernel
from .. import mean as _mean
from .. import params as _params
from .gp import GP, _ptr


def sparsify(gp: GP, X, max_points: int, return_removed: bool = False):
    """Indices (ascending) of the samples model::SparsifiedGP::_sparsify keeps out of the rows of X, computed with gp's
    device handle and workspace.  With return_removed, also the removal order and the density at each removal."""
    X = np.ascontiguousarray(np.atleast_2d(X), dtype=np.float64)
    N, D = X.shape
    keep = np.empty(min(N, max_points) if max_points >= 0 else 0, dtype=np.int64)
    R = max(N - max_points, 0)
    rem = np.empty(R, dtype=np.int64) if return_removed else None
    dens = np.empty(R) if return_removed else None
    _lib.check(gp._lib.lb_sparsify(gp._h, N, D, _ptr(X), max_points, _ptr(keep),
                                   _ptr(rem) if return_removed and R else None, _ptr(dens) if return_removed and R else None),
               "lb_sparsify")
    return (keep, rem, dens) if return_removed else keep


class SparsifiedGP(GP):
    def __init__(self, dim_in: int = -1, dim_out: int = -1, params=None, kernel=_kernel.MaternFiveHalves, mean=_mean.Data,
                 hp_opt=None, device: int = 0, precision: str = "fp64"):
        self._max_points = int(_params.get(params, "model_sparse_gp", "max_points"))
        if dim_in > 0:
            self._check_cap(dim_in)
        super().__init__(dim_in, dim_out, params=params, kernel=kernel, mean=mean, hp_opt=hp_opt, device=device,
                         precision=precision)

    def max_points(self) -> int:
        return self._max_points

    def _check_cap(self, dim: int) -> None:
        # with max_points < D the reference's partial_sort reads past the row (undefined behaviour)
        if self._max_points < dim:
            raise ValueError(f"model_sparse_gp.max_points = {self._max_points} is smaller than the input dimension {dim}")

    def copy(self) -> "SparsifiedGP":
        g = GP.copy(self)
        g.__class__ = SparsifiedGP
        return g

    # ---- sparsified_gp.hpp:84-101 ----
    def compute(self, samples, observations, compute_kernel: bool = True) -> None:
        assert len(samples) != 0 and len(observations) != 0 and len(samples) == len(observations)
        if len(samples) <= self._max_points:
            return GP.compute(self, samples, observations, compute_kernel)
        X = np.array(samples, dtype=np.float64, order="C")
        Y = np.array(observations, dtype=np.float64, order="C")
        if X.ndim == 1:
            X = X[:, None]
        if Y.ndim == 1:
            Y = Y[:, None]
        self._check_cap(X.shape[1])
        keep = sparsify(self, X, self._max_points)
        GP.compute(self, X[keep], Y[keep], compute_kernel)

    # ---- sparsified_gp.hpp:105-119 ----
    def add_sample(self, sample, observation) -> None:
        if len(self._samples) + 1 <= self._max_points:
            return GP.add_sample(self, sample, observation)
        # past the cap the reference appends, then re-sparsifies the current samples plus the new one and refits from
        # scratch: only that refit is observable, so the append is skipped
        sample = np.atleast_1d(np.asarray(sample, dtype=np.float64))
        observation = np.atleast_1d(np.asarray(observation, dtype=np.float64))
        assert sample.size == self._dim_in
        assert observation.size == self._dim_out
        X = np.vstack([self._sample_matrix(), sample[None, :]])
        Y = np.vstack([self._observations, observation[None, :]])
        self.compute(X, Y, True)
