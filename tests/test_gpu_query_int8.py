"""The panel query's trailing update as int8 digit products on tcgen05 (query_i8.cu) against the DMMA update it replaces:
same mu bit for bit (mu does not go through the update), sigma^2 within 1e-12, deterministic and independent of the batch
order, the cached digit planes of L follow every change of the factor, clones share them, and super-blocks beyond the
kernel's K bound take the DMMA update."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TOL_S2 = 1e-12


def _gp(N, D=6, noise=0.01, seed=1234):
    from limbo_b200 import kernel, mean, model, synth

    class Prm:
        class kernel:
            pass
    Prm.kernel.noise = noise
    X = synth.points(seed, N, D)
    y = synth.targets(X)
    gp = model.GP(D, 1, params=Prm, kernel=kernel.SquaredExpARD, mean=mean.Data)
    gp.compute(list(X), list(y[:, None]))
    return gp, X


def _queries(X, M=1500, D=6):
    from limbo_b200 import synth
    # candidates plus training points (sigma^2 ~ noise: the worst case for the truncated digit products)
    return np.concatenate([synth.points(1235, M, D), X[:256]])


def _run(gp, Xq, on, max_k=0):
    from limbo_b200 import _lib
    lib = _lib.load()
    lib.lb_debug_set_query_int8(on, max_k)
    try:
        return gp.query_batch(Xq)
    finally:
        lib.lb_debug_set_query_int8(-1, 0)


def _check(a, b):
    mu_a, s2_a = a
    mu_b, s2_b = b
    assert np.array_equal(mu_a, mu_b)
    d = np.abs(s2_a - s2_b).max()
    assert d <= TOL_S2, d


@pytest.mark.parametrize("N", [4096, 8192, 16384])
def test_int8_update_matches_dmma(N):
    gp, X = _gp(N)
    Xq = _queries(X)
    i8 = _run(gp, Xq, 1)
    dm = _run(gp, Xq, 0)
    _check(i8, dm)
    assert np.all(i8[1] > 0)


def test_int8_deterministic_and_order_independent():
    gp, X = _gp(8192)
    Xq = _queries(X)
    mu, s2 = _run(gp, Xq, 1)
    mu2, s22 = _run(gp, Xq, 1)
    assert np.array_equal(mu, mu2) and np.array_equal(s2, s22)
    perm = np.random.default_rng(0).permutation(len(Xq))
    mu3, s23 = _run(gp, Xq[perm], 1)
    assert np.array_equal(mu3, mu[perm]) and np.array_equal(s23, s2[perm])


def test_int8_planes_follow_the_factor():
    from limbo_b200 import synth
    gp, X = _gp(4096 + 128)
    Xq = _queries(X)
    s2_0 = _run(gp, Xq, 1)[1]
    # new hyper-parameters, refit
    gp.kernel_function().set_h_params(gp.kernel_function().h_params() - 0.2)
    gp.recompute(False)
    a = _run(gp, Xq, 1)
    _check(a, _run(gp, Xq, 0))
    assert np.abs(a[1] - s2_0).max() > 1e-6
    # incremental update of the factor (one more sample)
    x = synth.points(99, 1, 6)[0]
    gp.add_sample(x, np.array([0.3]))
    b = _run(gp, Xq, 1)
    _check(b, _run(gp, Xq, 0))
    # hyper-parameters set back, full recompute
    gp.kernel_function().set_h_params(gp.kernel_function().h_params() + 0.2)
    gp.recompute(True)
    _check(_run(gp, Xq, 1), _run(gp, Xq, 0))


def test_int8_clone_shares_planes():
    gp, X = _gp(8192)
    Xq = _queries(X)
    ref = _run(gp, Xq, 1)          # builds the digit planes of the source
    cl = gp.copy()                 # shares L and the planes
    a = _run(cl, Xq, 1)
    assert np.array_equal(a[0], ref[0]) and np.array_equal(a[1], ref[1])
    # the source refits: its planes are rebuilt in a buffer of its own, the clone keeps answering for the old factor
    gp.kernel_function().set_h_params(gp.kernel_function().h_params() - 0.2)
    gp.recompute(False)
    _check(_run(gp, Xq, 1), _run(gp, Xq, 0))
    b = _run(cl, Xq, 1)
    assert np.array_equal(b[0], ref[0]) and np.array_equal(b[1], ref[1])


def test_int8_k_bound_guard():
    """Super-blocks whose K range exceeds the bound take the DMMA update; a bound above the exactness limit is ignored."""
    gp, X = _gp(8192)
    Xq = _queries(X)
    dm = _run(gp, Xq, 0)
    full = _run(gp, Xq, 1)
    mixed = _run(gp, Xq, 1, max_k=4096)  # super-blocks 1 and 2 on int8, 3 on DMMA
    _check(mixed, dm)
    assert not np.array_equal(mixed[1], full[1]) or not np.array_equal(mixed[1], dm[1])
    over = _run(gp, Xq, 1, max_k=1 << 20)
    assert np.array_equal(over[1], full[1])
