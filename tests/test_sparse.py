"""CPU checks of the SparsifiedGP pieces that need no GPU: the literal restatement of SparsifiedGP::_sparsify
(oracle/sparse_literal.cpp) reproduces the reference's own kept sets (tests/golden/sparse/), the reference itself does
where it is built, lb_sparsify is exported, and SparsifiedGP rejects a cap below the input dimension."""
import glob
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "sparse", "*.npz")))
IDS = [os.path.basename(p)[:-4] for p in GOLD]


def literal_keep(X, max_points, n0=0):
    """kept indices after compute(X[:n0]) and add_sample for the rest (n0 = 0: one compute), by the literal restatement"""
    from oracle import sparse
    if not n0:
        return sparse.sparsify(X, max_points)[0]
    keep = np.arange(n0) if n0 <= max_points else sparse.sparsify(X[:n0], max_points)[0]
    for i in range(n0, len(X)):
        keep = np.append(keep, i)
        if len(keep) > max_points:
            keep = keep[sparse.sparsify(X[keep], max_points)[0]]
    return keep


def test_fixtures_present():
    assert len(GOLD) == 8


@pytest.mark.parametrize("path", GOLD, ids=IDS)
def test_literal_restatement_reproduces_reference(path):
    g = np.load(path)
    keep = literal_keep(g["X"], int(g["max_points"]), int(g["n0"]))
    assert np.array_equal(keep, g["keep"])


@pytest.mark.parametrize("path", GOLD, ids=IDS)
def test_reference_build_agrees_with_fixtures(path):
    from oracle import sparse
    if not os.path.exists(sparse.REF_LIB_PATH):
        pytest.skip("oracle/_ref/libref_sparse.so not built (needs the reference's sources at build time)")
    g = np.load(path)
    r = sparse.ref_run(g["X"], int(g["max_points"]), n0=int(g["n0"]))
    assert np.array_equal(r["keep"], g["keep"])


def test_ties_and_duplicates_take_lowest_index():
    from oracle import sparse
    # D = 1: the closest pair always has equal densities; x = 0, 1, 1.5, 3: the pair (1, 1.5) ties, index 1 goes first
    keep, rem, dens = sparse.sparsify(np.array([[0.0], [1.0], [1.5], [3.0]]), 3)
    assert rem.tolist() == [1] and dens.tolist() == [0.5] and keep.tolist() == [0, 2, 3]
    # exact copies: density 0 for both, the lower index goes
    keep, rem, _ = sparse.sparsify(np.array([[0.0, 0.0], [2.0, 1.0], [5.0, 5.0], [2.0, 1.0], [9.0, 0.0]]), 4)
    assert rem.tolist() == [1]


def test_lb_sparsify_exported(lib):
    from limbo_b200 import _lib
    assert hasattr(lib, "lb_sparsify") and "lb_sparsify" in _lib.DECLARED_SYMBOLS


def test_cap_below_dimension_rejected():
    from limbo_b200 import model

    class Prm:
        class model_sparse_gp:
            max_points = 2
    with pytest.raises(ValueError, match="max_points"):
        model.SparsifiedGP(3, 1, params=Prm)
    from oracle import sparse
    with pytest.raises(ValueError):
        sparse.sparsify(np.zeros((5, 3)), 2)


def test_default_cap_is_the_reference_default():
    from limbo_b200 import params
    assert params.get(None, "model_sparse_gp", "max_points") == 200
