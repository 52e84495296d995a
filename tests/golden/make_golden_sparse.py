"""Generates tests/golden/sparse/*.npz by running the REFERENCE'S OWN model::SparsifiedGP and model::MultiGP over it
(oracle/_ref/libref_sparse.so = /root/reference/src/limbo headers compiled against the Eigen stand-in, see
oracle/ref_sparse/) on seeded inputs.  Run where the reference's sources exist:   python tests/golden/make_golden_sparse.py
The fixtures pin the kept set (ties included: the lowest index wins), mean::Data over the kept observations, the
add_sample re-sparsification and the hyper-parameters after Rprop on the kept samples."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from limbo_b200 import synth  # noqa: E402
from oracle import sparse  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "sparse")

CASES = [
    # name, kernel_id (0 SE-ARD, 1 Matern-5/2), N, D, P, max_points, M, n0 (add_sample start), rprop_iters, multi, duplicated blocks
    ("se_ard_n100_d1_m33", 0, 100, 1, 1, 33, 16, 0, 0, False, False),  # the reference's test_sparse_gp configuration
    ("matern52_n300_d2_m64", 1, 300, 2, 1, 64, 16, 0, 0, False, False),
    ("matern52_n500_d6_m200", 1, 500, 6, 1, 200, 16, 0, 0, False, False),
    ("matern52_n240_d3_m40_dup", 1, 240, 3, 1, 40, 16, 0, 0, False, True),
    ("matern52_n80_d6_m6", 1, 80, 6, 1, 6, 16, 0, 0, False, False),  # max_points == D
    ("matern52_n70_d2_m50_add10", 1, 70, 2, 1, 50, 16, 60, 0, False, False),
    ("se_ard_n120_d2_m50_rprop5", 0, 120, 2, 1, 50, 8, 0, 5, False, False),
    ("multi_matern52_n150_d2_p2_m40", 1, 150, 2, 2, 40, 16, 0, 0, True, False),
]

os.makedirs(OUT, exist_ok=True)
for name, kid, N, D, P, m, M, n0, iters, multi, dup in CASES:
    X = synth.points(4321 + N, N, D)
    if dup:  # blocks of exact copies: every copy has the density of its original, so ties decide
        X[N // 2:N // 2 + N // 4] = X[:N // 4]
        X[-N // 8:] = X[N // 4:N // 4 + N // 8]
    y = synth.targets(X)
    Y = np.stack([y * (p + 1) + 0.1 * p for p in range(P)], axis=1)
    Xq = synth.points(4322 + N, M, D)
    r = sparse.ref_run(X, m, Y=Y, kernel_id=kid, n0=n0, Xq=Xq, rprop_iters=iters, multi=multi)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), kernel_id=kid, max_points=m, n0=n0, rprop_iters=iters, multi=multi,
                        noise=0.01, X=X, Y=Y, Xq=Xq, keep=r["keep"], mu=r["mu"], sigma2=r["sigma2"], hp=r["hp"])
    print(name, "kept", len(r["keep"]))
