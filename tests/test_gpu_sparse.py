"""SparsifiedGP on the GPU: lb_sparsify (limbo_b200/csrc/sparsify.cu) against the reference's own kept sets
(tests/golden/sparse/) and the literal restatement of SparsifiedGP::_sparsify (oracle/sparse_literal.cpp) — kept sets
AND removal orders identical, ties included — then the fitted model against the reference's predictions, MultiGP over
SparsifiedGP, a full-size trace check against an independent torch recomputation, the launch count, the buffer pool and
an external stream."""
import numpy as np
import pytest

from test_sparse import GOLD, IDS, literal_keep

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def handle():
    """a model whose device handle and workspace run the selections"""
    import __graft_entry__ as g
    g.build()
    from limbo_b200 import model
    return model.GP(1, 1)


def _points(seed, N, D, dup=False):
    from limbo_b200 import synth
    X = synth.points(seed, N, D)
    if dup:
        X[N // 2:N // 2 + N // 4] = X[:N // 4]
        X[-N // 8:] = X[N // 4:N // 4 + N // 8]
    return X


@pytest.mark.parametrize("path", GOLD, ids=IDS)
def test_fixture_kept_set_and_removal_order(path, handle):
    from limbo_b200.model import sparsify
    from oracle import sparse
    g = np.load(path)
    X, m, n0 = g["X"], int(g["max_points"]), int(g["n0"])
    if n0:  # the add_sample sequence: one re-sparsification of max_points + 1 samples per call
        keep = np.arange(n0) if n0 <= m else sparsify(handle, X[:n0], m)
        for i in range(n0, len(X)):
            keep = np.append(keep, i)
            if len(keep) > m:
                k, rem, dens = sparsify(handle, X[keep], m, return_removed=True)
                ko, remo, denso = sparse.sparsify(X[keep], m)
                assert np.array_equal(rem, remo) and np.array_equal(dens, denso)
                keep = keep[k]
        assert np.array_equal(keep, g["keep"])
        return
    keep, rem, dens = sparsify(handle, X, m, return_removed=True)
    assert np.array_equal(keep, g["keep"])
    ko, remo, denso = sparse.sparsify(X, m)
    assert np.array_equal(rem, remo)
    assert np.array_equal(dens, denso)  # bit for bit


SWEEP = []
for D in (1, 2, 3, 6, 12, 64):
    N = 400
    for cap in sorted({D, max(D, 50), max(D, N // 8), N - 1, N + 3}):
        SWEEP.append((N, D, cap, D in (3, 12)))
SWEEP += [(2048, 6, 256, False), (2048, 1, 1, False), (2048, 3, 1024, True), (1000, 2, 2, True)]


@pytest.mark.parametrize("N,D,cap,dup", SWEEP, ids=[f"n{n}_d{d}_m{c}{'_dup' if u else ''}" for n, d, c, u in SWEEP])
def test_sweep_against_literal_restatement(N, D, cap, dup, handle):
    from limbo_b200.model import sparsify
    from oracle import sparse
    X = _points(1000 + 7 * D + N, N, D, dup)
    keep, rem, dens = sparsify(handle, X, cap, return_removed=True)
    ko, remo, denso = sparse.sparsify(X, cap)
    assert np.array_equal(keep, ko)
    assert np.array_equal(rem, remo)
    assert np.array_equal(dens, denso)


def _model_for(g):
    from limbo_b200 import kernel, mean, model, opt
    iters = int(g["rprop_iters"])

    class Prm:
        class kernel:
            noise = float(g["noise"])
            optimize_noise = False

        class opt_rprop:
            iterations = max(iters, 1)
            eps_stop = 0.0

        class model_sparse_gp:
            max_points = int(g["max_points"])
    kern = kernel.SquaredExpARD if int(g["kernel_id"]) == 0 else kernel.MaternFiveHalves
    X, Y = g["X"], g["Y"]
    if bool(g["multi"]):
        return model.MultiGP(X.shape[1], Y.shape[1], params=Prm, kernel=kern, mean=mean.Data, gp=model.SparsifiedGP)
    return model.SparsifiedGP(X.shape[1], Y.shape[1], params=Prm, kernel=kern, mean=mean.Data,
                              hp_opt=model.KernelLFOpt(Prm, opt.Rprop(Prm)))


@pytest.mark.parametrize("path", GOLD, ids=IDS)
def test_sparsified_gp_matches_reference_predictions(path):
    g = np.load(path)
    X, Y, Xq, n0, iters = g["X"], g["Y"], g["Xq"], int(g["n0"]), int(g["rprop_iters"])
    gp = _model_for(g)
    if n0:
        gp.compute(X[:n0], Y[:n0])
        for i in range(n0, len(X)):
            gp.add_sample(X[i], Y[i])
    else:
        gp.compute(X, Y)
    if bool(g["multi"]):
        for sub in gp.gp_models():
            assert np.array_equal(np.stack(sub.samples()), X[g["keep"]])
        mu, s2 = gp.query_batch(Xq)
        assert np.abs(mu - g["mu"]).max() <= 1e-10 and np.abs(s2 - g["sigma2"]).max() <= 1e-10
        assert gp.nb_samples() == len(X)
        return
    assert np.array_equal(np.stack(gp.samples()), X[g["keep"]])
    assert np.array_equal(gp.observations_matrix(), Y[g["keep"]])
    if iters:
        gp.optimize_hyperparams()
        assert np.abs(gp.kernel_function().h_params() - g["hp"]).max() <= 1e-9
    mu, s2 = gp.query_batch(Xq)
    assert np.abs(mu - g["mu"]).max() <= 1e-10 and np.abs(s2 - g["sigma2"]).max() <= 1e-10
    c = gp.copy()
    assert type(c).__name__ == "SparsifiedGP" and c.max_points() == gp.max_points()


def _torch_densities(Xt, live, D):
    """density of every live row over the live set: plain elementwise fp64 torch ops in the reference's operation order
    (differences, squares, sum from 0 in order d = 0..D-1, sqrt), D smallest by topk (sorted), added in ascending order"""
    import torch
    idx = torch.nonzero(live).squeeze(1)
    Xl = Xt[idx]
    n = Xl.shape[0]
    dens = torch.empty(n, dtype=torch.float64, device=Xt.device)
    for r0 in range(0, n, 1024):
        r1 = min(n, r0 + 1024)
        s = torch.zeros((r1 - r0, n), dtype=torch.float64, device=Xt.device)
        for d in range(D):
            t = Xl[r0:r1, d:d + 1] - Xl[:, d][None, :]
            s = s + t * t
        dist = torch.sqrt(s)
        dist[torch.arange(r1 - r0, device=Xt.device), torch.arange(r0, r1, device=Xt.device)] = float("inf")
        v = torch.topk(dist, D, dim=1, largest=False, sorted=True).values
        acc = torch.zeros(r1 - r0, dtype=torch.float64, device=Xt.device)
        for r in range(D):
            acc = acc + v[:, r]
        dens[r0:r1] = acc
    return idx, dens


def test_full_size_trace_and_constant_launch_count(handle):
    import torch
    from limbo_b200.model import sparsify
    N, D = 16384, 6
    X = _points(99, N, D)
    l0 = handle.launch_count()
    keep, rem, dens = sparsify(handle, X, 2048, return_removed=True)
    l1 = handle.launch_count()
    keep2 = sparsify(handle, X, 8192)
    l2 = handle.launch_count()
    assert l1 - l0 == l2 - l1 <= 2, (l1 - l0, l2 - l1)
    assert len(keep) == 2048 and len(rem) == N - 2048 and np.array_equal(np.sort(np.concatenate([keep, rem])), np.arange(N))
    assert set(keep) <= set(keep2)  # the greedy order is a prefix: the first N - 8192 removals are shared
    Xt = torch.tensor(X, dtype=torch.float64, device="cuda")
    rng = np.random.default_rng(5)
    steps = sorted(set([0, 1, len(rem) - 1] + rng.choice(len(rem), 29, replace=False).tolist()))
    for t in steps:
        live = torch.ones(N, dtype=torch.bool, device="cuda")
        live[torch.tensor(rem[:t], dtype=torch.long, device="cuda")] = False
        idx, d = _torch_densities(Xt, live, D)
        m = torch.min(d)
        k = int(idx[torch.nonzero(d == m)[0, 0]])  # lowest index among the minima
        assert rem[t] == k, (t, rem[t], k)
        assert dens[t] == float(m), (t, dens[t], float(m))


def test_pool_reuse_and_external_stream(handle):
    import torch
    from limbo_b200 import _lib
    from limbo_b200.model import sparsify
    X = _points(5, 3000, 4)
    ref = sparsify(handle, X, 300, return_removed=True)
    lib = _lib.load()
    before = lib.lb_debug_pool_mallocs()
    again = sparsify(handle, X, 300, return_removed=True)
    assert lib.lb_debug_pool_mallocs() == before
    s = torch.cuda.Stream()
    handle.set_stream(s.cuda_stream)
    try:
        on_stream = sparsify(handle, X, 300, return_removed=True)
    finally:
        handle.set_stream(None)
    for a, b, c in zip(ref, again, on_stream):
        assert np.array_equal(a, b) and np.array_equal(a, c)


def test_arguments_and_identity(handle):
    from limbo_b200 import _lib
    from limbo_b200.model import sparsify
    X = _points(3, 50, 4)
    l0 = handle.launch_count()
    assert np.array_equal(sparsify(handle, X, 50), np.arange(50)) and np.array_equal(sparsify(handle, X, 80), np.arange(50))
    assert handle.launch_count() == l0
    with pytest.raises(_lib.LimboB200Error, match="LB_ERR_ARG"):
        sparsify(handle, X, 3)
    with pytest.raises(_lib.LimboB200Error, match="LB_ERR_ARG"):
        sparsify(handle, np.zeros((10, 65)), 100)
