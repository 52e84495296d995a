"""Generates tests/golden/restatement/*.npz from the REFERENCE'S OWN code (oracle/_ref/libref_gp.so, see make_golden.py):
the cases tests/test_oracle_vs_ref.py pins the oracle restatement with.
 * k<kernel>_n<N>_d<D>_p<P> : GP::compute, query, compute_log_lik, compute_kernel_grad_log_lik  (gp.hpp:88, 159, 267, 285)
 * rprop_n50_d2             : KernelLFOpt<Rprop>, 10 iterations                                (model/gp/kernel_lf_opt.hpp)
 * incremental_n40_d2       : 25 samples, then 15 add_sample calls                             (gp.hpp:126)
K and L are stored as a seeded sample of rows (always including the last one) to keep the fixtures small.
Run where the reference's sources are available:   python tests/golden/make_golden_restatement.py"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from limbo_b200 import synth  # noqa: E402
from oracle import ref  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "restatement")
os.makedirs(OUT, exist_ok=True)
ROWS = 10


def sample_rows(N: int, seed: int) -> np.ndarray:
    if N <= ROWS:
        return np.arange(N)
    rows = np.random.default_rng(seed).choice(N - 1, ROWS - 1, replace=False)
    return np.sort(np.append(rows, N - 1))


def save(name, **arrays):
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **arrays)
    print(name, "ok")


for kid in (0, 1, 2, 3):
    for N, D, P in ((5, 1, 1), (33, 3, 2), (120, 6, 1)):
        rng = np.random.default_rng(100 * kid + N)
        hp = rng.uniform(-0.7, 0.7, D + 1 if kid == 0 else 2)
        X = synth.points(77 + N, N, D)
        y = synth.targets(X)
        Y = np.stack([y * (p + 1) - 0.3 * p for p in range(P)], axis=1)
        Xq = synth.points(78, 25, D)
        r = ref.run(kid, X, Y, 0.015, hp=hp, Xq=Xq)
        rows = sample_rows(N, kid * 1000 + N)
        save(f"k{kid}_n{N}_d{D}_p{P}", kernel_id=kid, noise=0.015, hp=hp, X=X, Y=Y, Xq=Xq, rows=rows, K_rows=r["K"][rows],
             L_rows=r["L"][rows], alpha=r["alpha"], mu=r["mu"], sigma2=r["sigma2"], loglik=r["loglik"], grad=r["grad"])

X = synth.points(5, 50, 2)
y = synth.targets(X)
save("rprop_n50_d2", kernel_id=0, noise=0.01, rprop_iters=10, X=X, Y=y[:, None], hp=ref.run(0, X, y, 0.01, rprop_iters=10)["hp"])

X = synth.points(6, 40, 2)
y = synth.targets(X)[:, None]
r = ref.run(1, X, y, 0.01, n0=25)
rows = sample_rows(40, 40)
save("incremental_n40_d2", kernel_id=1, noise=0.01, n0=25, X=X, Y=y, rows=rows, L_rows=r["L"][rows], alpha=r["alpha"])
