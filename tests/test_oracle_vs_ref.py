"""Pins the oracle restatement against the reference ITSELF: tests/golden/restatement/ holds what the reference's own
headers, compiled against the Eigen/Boost stand-in (oracle/ref_shim), computed on these inputs
(tests/golden/make_golden_restatement.py).  K and L are compared on a seeded sample of rows."""
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "restatement")


def _gold(name):
    return np.load(os.path.join(GOLD, name + ".npz"))


@pytest.mark.parametrize("kid", [0, 1, 2, 3])
@pytest.mark.parametrize("N,D,P", [(5, 1, 1), (33, 3, 2), (120, 6, 1)])
def test_restatement_equals_reference(oracle_mod, kid, N, D, P):
    O = oracle_mod
    r = _gold(f"k{kid}_n{N}_d{D}_p{P}")
    X, Y, Xq, rows = r["X"], r["Y"], r["Xq"], r["rows"]
    og = O.OracleGP()
    og.set_data(X, Y - Y.mean(axis=0))
    og.set_kernel(kid, r["hp"], float(r["noise"]))
    assert og.fit() == -1
    assert np.abs(og.get(0)[rows] - r["K_rows"]).max() <= 1e-15
    assert np.abs(og.get(1)[rows] - r["L_rows"]).max() <= 1e-12
    assert np.abs(og.get(2) - r["alpha"]).max() <= 1e-11 * np.abs(r["alpha"]).max()
    mu, s2 = og.query(Xq)
    assert np.abs(mu + Y.mean(axis=0) - r["mu"]).max() <= 1e-12
    assert np.abs(s2 - r["sigma2"]).max() <= 1e-13
    assert abs(og.log_lik() - r["loglik"]) <= 1e-12 * abs(r["loglik"])
    assert np.abs(og.grad() - r["grad"]).max() <= 1e-10 * max(1.0, np.abs(r["grad"]).max())


def test_rprop_trajectory_equals_reference(oracle_mod):
    """KernelLFOpt<Rprop> in the reference vs the restated Rprop on the restated objective."""
    O = oracle_mod
    r = _gold("rprop_n50_d2")
    X, Y = r["X"], r["Y"]
    og = O.OracleGP()
    og.set_data(X, Y - Y.mean())
    og.set_kernel(0, np.zeros(3), float(r["noise"]))
    og.fit()
    best, ne = og.rprop_lml(np.zeros(3), int(r["rprop_iters"]))
    assert ne == 10 and np.abs(best - r["hp"]).max() <= 1e-12


def test_incremental_equals_reference(oracle_mod):
    O = oracle_mod
    r = _gold("incremental_n40_d2")
    X, y, n0, rows = r["X"], r["Y"], int(r["n0"]), r["rows"]
    og = O.OracleGP()
    og.set_data(X[:n0], y[:n0] - y[:n0].mean())
    og.set_kernel(1, np.zeros(2), float(r["noise"]))
    og.fit()
    for i in range(n0, X.shape[0]):
        og.append(X[i], y[: i + 1] - y[: i + 1].mean())
    assert np.abs(og.get(1)[rows] - r["L_rows"]).max() <= 1e-12
    assert np.abs(og.get(2) - r["alpha"]).max() <= 1e-11 * np.abs(r["alpha"]).max()
