"""Timing of SparsifiedGP's selection (lb_sparsify, limbo_b200/csrc/sparsify.cu) and of the whole SparsifiedGP.compute,
next to the reference's own SparsifiedGP::compute (oracle/_ref/libref_sparse.so, single host thread) at the sizes where
it finishes in minutes.  Writes one JSON file (default profiles/r03_sparsify.json).

    python tools/sparsify_timing.py [--out FILE] [--ref-sizes 1024,2048] [--skip-65536]

GPU times are CUDA events on the handle's stream around one call after a warm-up call of the same shape (the call ends
with a device-to-host copy of the result, so the events bracket the whole selection); the card's name and power limit
are read in the same run.  Inputs are synth.points (uniform in [0, 1]^D), D = 6."""
import argparse
import json
import os
import platform
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def cpu_name():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return platform.processor()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_sparsify.json"))
    ap.add_argument("--ref-sizes", default="1024,2048")
    ap.add_argument("--skip-65536", action="store_true")
    a = ap.parse_args()
    import torch
    from limbo_b200 import kernel, mean, model, synth
    from limbo_b200.model import sparsify
    D = 6
    res = {"card": card(), "D": D, "gpu": [], "reference": [], "compute": []}
    gp = model.GP(D, 1)
    stream = torch.cuda.Stream()
    gp.set_stream(stream.cuda_stream)
    sizes = [4096, 16384] + ([] if a.skip_65536 else [65536])
    for N in sizes:
        X = synth.points(2024 + N, N, D)
        for cap in (200, 2048):
            sparsify(gp, X, cap)  # warm-up, same shape
            l0 = gp.launch_count()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            sparsify(gp, X, cap)
            e1.record(stream)
            e1.synchronize()
            ms = e0.elapsed_time(e1)
            rec = {"N": N, "max_points": cap, "removals": N - cap, "ms": ms, "us_per_removal": 1e3 * ms / (N - cap),
                   "launches": gp.launch_count() - l0}
            res["gpu"].append(rec)
            print(json.dumps(rec), flush=True)
    gp.set_stream(None)

    # the trade a user makes: fit all 16384 samples, or select 2048 and fit those (host clock; both end in a device sync)
    N = 16384
    X = synth.points(77, N, D)
    y = synth.targets(X)[:, None]

    class Prm:
        class model_sparse_gp:
            max_points = 2048
    for name, cls in (("GP.compute N=16384", model.GP), ("SparsifiedGP.compute 16384 -> 2048", model.SparsifiedGP)):
        m = cls(D, 1, params=Prm, kernel=kernel.MaternFiveHalves, mean=mean.Data)
        m.compute(X, y)  # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        m.compute(X, y)
        m.query_batch(X[:1])  # ends in a device sync
        rec = {"what": name, "s": time.perf_counter() - t0, "kept": m.nb_samples()}
        res["compute"].append(rec)
        print(json.dumps(rec), flush=True)

    from oracle import sparse
    if os.path.exists(sparse.REF_LIB_PATH) and a.ref_sizes:
        for N in [int(s) for s in a.ref_sizes.split(",")]:
            X = synth.points(2024 + N, N, D)
            r = sparse.ref_run(X, 200, Y=synth.targets(X)[:, None], want_keep=False)
            rec = {"N": N, "max_points": 200, "s": r["seconds"], "cpu": cpu_name(), "threads": 1}
            res["reference"].append(rec)
            print(json.dumps(rec), flush=True)
        if res["reference"]:
            last = res["reference"][-1]
            res["reference_extrapolated_16384"] = {
                "s": last["s"] * (16384 / last["N"]) ** 3, "note": f"EXTRAPOLATION from N={last['N']} by N^3, not measured"}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
