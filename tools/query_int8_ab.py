"""A/B of the panel query's trailing update: int8 digit products on tcgen05 (LB_QUERY_INT8=1, the default) against the DMMA
update (LB_QUERY_INT8=0), on the flagship workload of bench.py (N = 16384, D = 6, SE-ARD, M = 10^4 UCB candidates).

Each round runs one process per mode, modes alternating.  A process times with CUDA events
  - the query alone (lb_acq_argmax_dev on a fitted model; the digit planes of L are cached after the first query), and
  - the whole bench step (set_data, set_kernel, fit, acq_argmax: the planes are rebuilt after every fit),
and stores mu / sigma^2 of the candidates plus 256 training points (the worst case, sigma^2 ~ noise).  The parent compares
the outputs of the two modes, reports medians and spreads with the card name and power limit, and writes
profiles/r04_query_int8.json (or --out).

usage: python tools/query_int8_ab.py [--rounds 3] [--reps 10] [--out PATH]"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def child(out_dir: str, reps: int) -> None:
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from limbo_b200 import _lib, kernel, mean, model, synth
    n, d, m = bench.N_TRAIN, bench.DIM, bench.M_CAND
    X = synth.points(1234, n, d)
    y = synth.targets(X)
    Xq = synth.points(1235, m, d)
    st = torch.cuda.Stream()
    torch.cuda.set_stream(st)
    kcls = getattr(kernel, bench.KERNEL_NAME)
    gp = model.GP(d, 1, kernel=kcls, mean=mean.Data)
    gp.set_stream(st.cuda_stream)
    lib = _lib.load()
    h = gp._h
    dev = torch.device("cuda")
    dX, dY = torch.from_numpy(X).to(dev), torch.from_numpy(y - y.mean()).to(dev)
    dXq = torch.from_numpy(Xq).to(dev)
    dB, dI = torch.zeros(1, dtype=torch.float64, device=dev), torch.zeros(1, dtype=torch.int64, device=dev)
    ap = np.array([bench.UCB_ALPHA, 0.0])
    hp = np.zeros(d + 1)

    def fit():
        _lib.check(lib.lb_set_data_dev(h, n, d, 1, dX.data_ptr(), dY.data_ptr()), "set_data_dev")
        _lib.check(lib.lb_set_kernel(h, kcls.kernel_id, hp.ctypes.data, hp.size, bench.NOISE), "set_kernel")
        _lib.check(lib.lb_fit_async(h), "fit_async")

    def query():
        _lib.check(lib.lb_acq_argmax_dev(h, 0, ap.ctypes.data, m, dXq.data_ptr(), None, float(y.mean()), None, dB.data_ptr(),
                                         dI.data_ptr()), "acq_argmax_dev")

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        out = []
        for _ in range(reps):
            e0.record(st)
            fn()
            e1.record(st)
            torch.cuda.synchronize()
            out.append(e0.elapsed_time(e1))
        return out

    def step():
        fit()
        query()

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    t_step = timed(step)
    t_query = timed(query)
    best = (float(dB.item()), int(dI.item()))
    # outputs on the same seeded inputs (host path of the same model)
    gp.compute(list(X), list(y[:, None]))
    mu, s2 = gp.query_batch(np.concatenate([Xq, X[:256]]))
    np.save(os.path.join(out_dir, "mu.npy"), np.asarray(mu, dtype=np.float64))
    np.save(os.path.join(out_dir, "s2.npy"), np.asarray(s2, dtype=np.float64))
    json.dump({"step_ms": t_step, "query_ms": t_query, "best": best}, open(os.path.join(out_dir, "t.json"), "w"))


def card() -> dict:
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60)
        name, pl, clk = [s.strip() for s in r.stdout.splitlines()[0].split(",")]
        return {"name": name, "power_limit": pl, "max_sm_clock": clk}
    except Exception as e:  # noqa: BLE001 - reported, not fatal
        return {"error": str(e)}


def stats(v):
    v = np.asarray(v, dtype=float)
    return {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max()), "n": int(v.size)}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_query_int8.json"))
    ap.add_argument("--child", default=None)
    a = ap.parse_args()
    if a.child:
        child(a.child, a.reps)
        return
    runs = {0: [], 1: []}
    outs = {}
    with tempfile.TemporaryDirectory() as tmp:
        for r in range(a.rounds):
            for mode in (0, 1):
                d = os.path.join(tmp, f"r{r}_m{mode}")
                os.makedirs(d)
                env = dict(os.environ, LB_QUERY_INT8=str(mode))
                subprocess.run([sys.executable, os.path.abspath(__file__), "--child", d, "--reps", str(a.reps)], env=env, check=True, cwd=ROOT)
                t = json.load(open(os.path.join(d, "t.json")))
                runs[mode].append(t)
                outs[(r, mode)] = (np.load(os.path.join(d, "mu.npy")), np.load(os.path.join(d, "s2.npy")))
                print(f"round {r} LB_QUERY_INT8={mode}: step {np.median(t['step_ms']):.2f} ms, query {np.median(t['query_ms']):.2f} ms, "
                      f"best {t['best']}", flush=True)
    res = {"workload": "N=16384 D=6 SE-ARD M=10000 UCB (bench.py flagship step)", "card": card(), "rounds": a.rounds, "reps": a.reps}
    for mode, key in ((0, "dmma"), (1, "int8")):
        step = [x for t in runs[mode] for x in t["step_ms"]]
        query = [x for t in runs[mode] for x in t["query_ms"]]
        res[key] = {"step_ms": stats(step), "query_ms": stats(query), "per_round_step_median": [float(np.median(t["step_ms"])) for t in runs[mode]],
                    "per_round_query_median": [float(np.median(t["query_ms"])) for t in runs[mode]], "best": runs[mode][-1]["best"]}
    mu0, s0 = outs[(0, 0)]
    mu1, s1 = outs[(0, 1)]
    res["outputs"] = {"mu_bit_equal": bool(np.array_equal(mu0, mu1)), "max_abs_dsigma2": float(np.abs(s0 - s1).max()),
                      "max_abs_dsigma2_training_points": float(np.abs(s0[-256:] - s1[-256:]).max()),
                      "same_best_index": runs[0][-1]["best"][1] == runs[1][-1]["best"][1],
                      "best_value_diff": abs(runs[0][-1]["best"][0] - runs[1][-1]["best"][0]),
                      "int8_run_to_run_bit_equal": all(np.array_equal(outs[(r, 1)][1], s1) for r in range(a.rounds))}
    res["speedup"] = {"query": res["dmma"]["query_ms"]["median"] / res["int8"]["query_ms"]["median"],
                      "step": res["dmma"]["step_ms"]["median"] / res["int8"]["step_ms"]["median"]}
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
