"""ctypes front-end of oracle/sparse_literal.cpp, the literal CPU restatement of model::SparsifiedGP::_sparsify.
TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "sparse_literal.cpp")
LIB_PATH = os.path.join(HERE, "_build", "libsparse_literal.so")
CXXFLAGS = ["-O3", "-fPIC", "-std=c++17", "-Wall", "-fno-fast-math", "-ffp-contract=off", "-pthread", "-shared"]

_lib = None


def build() -> str:
    if not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < os.path.getmtime(SRC):
        os.makedirs(os.path.dirname(LIB_PATH), exist_ok=True)
        subprocess.run(["g++", *CXXFLAGS, "-o", LIB_PATH, SRC], check=True, capture_output=True)
    return LIB_PATH


def load():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        vp = C.c_void_p
        _lib.sparse_literal.argtypes = [C.c_long, C.c_int, vp, C.c_long, vp, vp, vp, C.c_int]
        _lib.sparse_literal.restype = C.c_int
    return _lib


def sparsify(X, max_points: int, nthreads: int = 0):
    """(keep, removed, removed_density): kept original indices in ascending order, the removal order and the density of
    each removed point when it went."""
    X = np.ascontiguousarray(np.atleast_2d(X), dtype=np.float64)
    N, D = X.shape
    if N <= max_points:
        return np.arange(N, dtype=np.int64), np.zeros(0, np.int64), np.zeros(0)
    keep = np.empty(max_points, np.int64)
    rem = np.empty(N - max_points, np.int64)
    dens = np.empty(N - max_points)
    rc = load().sparse_literal(N, D, X.ctypes.data, max_points, keep.ctypes.data, rem.ctypes.data, dens.ctypes.data, nthreads)
    if rc != 0:
        raise ValueError(f"sparse_literal: error {rc} (N={N}, D={D}, max_points={max_points})")
    return keep, rem, dens


# ---- the reference's own model::SparsifiedGP (oracle/ref_sparse, built only where the reference's sources exist) ----
REF_LIB_PATH = os.path.join(HERE, "_ref", "libref_sparse.so")
REF_SRC = "/root/reference/src/limbo"

_ref = None


def ref_available() -> bool:
    return os.path.exists(REF_LIB_PATH) or os.path.isdir(REF_SRC)


def ref_build() -> str:
    if os.path.isdir(REF_SRC):
        subprocess.run(["make", "-C", os.path.join(HERE, "ref_sparse"), "CXX=g++"], check=True, capture_output=True)
    return REF_LIB_PATH


def ref_load():
    global _ref
    if _ref is None:
        if not os.path.exists(REF_LIB_PATH):
            ref_build()
        _ref = C.CDLL(REF_LIB_PATH)
        vp, lg, i, d = C.c_void_p, C.c_long, C.c_int, C.c_double
        _ref.ref_sparse_gp_run.argtypes = [i, lg, i, i, vp, vp, d, vp, i, lg, lg, lg, vp, i, i, vp, vp, vp, vp, vp, vp]
        _ref.ref_sparse_gp_run.restype = i
    return _ref


def ref_run(X, max_points: int, Y=None, kernel_id: int = 1, noise: float = 0.01, hp=None, n0: int = 0, Xq=None,
            rprop_iters: int = 0, multi: bool = False, want_keep: bool = True):
    """The reference's SparsifiedGP (or MultiGP over it, multi=True) with mean::Data: compute() on the first n0 samples
    then add_sample() for the rest (n0 = 0: one compute).  Returns a dict with keep (kept original indices), mu, sigma2,
    hp (kernel h-params after the optional Rprop) and seconds (wall time of the compute / add_sample sequence)."""
    lib = ref_load()
    X = np.ascontiguousarray(np.atleast_2d(X), dtype=np.float64)
    N, D = X.shape
    out = {}
    keep = np.zeros(N, np.int64) if want_keep else None
    nk = C.c_long(0)
    secs = C.c_double(0.0)
    if Y is not None:
        Y = np.ascontiguousarray(Y, dtype=np.float64).reshape(N, -1)
        P = Y.shape[1]
        Xq = np.zeros((0, D)) if Xq is None else np.ascontiguousarray(Xq, dtype=np.float64)
        M = Xq.shape[0]
        mu = np.zeros((M, P))
        s2 = np.zeros((M, P) if multi else M)
        nh = (D + 1) if kernel_id == 0 else 2
        hpa = None if hp is None else np.ascontiguousarray(hp, dtype=np.float64)
        hp_out = np.zeros(nh)
        rc = lib.ref_sparse_gp_run(kernel_id, N, D, P, X.ctypes.data, Y.ctypes.data, noise,
                                   None if hpa is None else hpa.ctypes.data, nh, max_points, n0, M, Xq.ctypes.data, rprop_iters,
                                   int(multi), None if keep is None else keep.ctypes.data, C.addressof(nk), mu.ctypes.data,
                                   s2.ctypes.data, hp_out.ctypes.data, C.addressof(secs))
        out.update(mu=mu, sigma2=s2, hp=hp_out, seconds=secs.value)
    else:
        rc = lib.ref_sparse_gp_run(kernel_id, N, D, 1, X.ctypes.data, None, noise, None, 0, max_points, n0, 0, None, 0, 0,
                                   keep.ctypes.data, C.addressof(nk), None, None, None, None)
    if rc != 0:
        raise RuntimeError(f"ref_sparse_gp_run: {rc}")
    if keep is not None:
        out["keep"] = keep[:nk.value].copy()
    return out
