#!/usr/bin/env python
"""bench.py — GP fit + batched query throughput on B200 (BASELINE.json's metric).

One "step" = one pass of the hot path over one batch of synthetic input:
    fit  : K-build (N x N) -> blocked Cholesky -> alpha            (model/gp.hpp:550-571)
    query: M UCB candidates: K*, L^-1 K*, mu, sigma^2, UCB, argmax (gp.hpp:159-167, acqui/ucb.hpp:83-90)
at N = 16384, D = 6, SquaredExpARD, fp64, M = 10000 (SURVEY.md §8d (i)).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload ...] [--dump-outputs DIR]

It runs from the tree as __graft_entry__.build() left it and writes nothing there (the tree may be read-only).

`value`   : steps/s with inputs already resident in HBM (device-pointer ABI), CUDA events on the library's stream.
`e2e`     : the same step through the public host API (limbo_b200.model.GP.compute + acqui.UCB.argmax_batch /
            dist.sharded_acq_argmax): host buffers in, host scalars out, copies inside the timed region.
N > 1     : STRONG scaling of the same global job.  The fit is DISTRIBUTED (limbo_b200/dist_fit.py: block-cyclic panel
            factorisation over the ranks, one panel broadcast per 256 columns, every rank assembles the complete factor from
            the messages; bit-identical to the single-GPU factor), then the 10^4 candidates are sharded over the ranks and one
            all_gather picks the argmax.  `limiter` names what bounds the step (--replicated-fit keeps the round-1 scheme:
            every rank refits alone).
`roofline`: the kernel with the largest share of the step, timed live with CUDA events around every launch
            (lb_profile_*); `roofline_kernels` is the per-kernel table.
`config4` / `config5`: sub-records for the two multi-GPU splits BASELINE.json names (1M EI candidates in tf32 sharded over
            the ranks; N = 65536 panel-broadcast Cholesky), measured in the same run at the same N.
`cpu_baseline` / `--impl reference`: the reference's own gp.hpp / ucb.hpp loops (oracle/_ref/libref_gp.so, compiled from
            /root/reference against the Eigen stand-in) when that library is present, else the oracle port; on the host
            cores, on a bounded sample extrapolated to the full size (stated in `sample`).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_TRAIN, DIM, M_CAND = 16384, 6, 10000
KERNEL_NAME = "SquaredExpARD"
WORKLOADS = {  # --workload: BASELINE.json configs that fit one GPU; the default is the configuration the metric is quoted on
    "n16384_se_ard": (16384, 6, 10000, "SquaredExpARD"),
    "config2_n4096_matern": (4096, 6, 10000, "MaternFiveHalves"),
}
NOISE = 0.01
UCB_ALPHA = 0.5
METRIC = "GP fit+query/s at N=16384,D=6 (fit = K-build+Cholesky+alpha, query = 10k UCB candidates+argmax, fp64)"
UNIT = "fit+query/s"
DATA = "synthetic (splitmix64 U[0,1)^D, Hartmann6 targets, deterministic)"


def workload_config(n_gpus: int) -> dict:
    per = -(-M_CAND // n_gpus)
    return {
        "workload": f"N={N_TRAIN}, D={DIM}, {KERNEL_NAME}, fp64, fit + {M_CAND} UCB queries + argmax (global job; candidates sharded over the GPUs)",
        "n_train": N_TRAIN, "dim": DIM, "kernel": KERNEL_NAME, "noise": NOISE,
        "global_candidates": M_CAND, "candidates_per_gpu": per,
        "parallelism": (f"fit distributed over {n_gpus} GPUs (1-D block-cyclic 256-column panels, one NCCL broadcast per panel, factor assembled on "
                        f"every rank), {M_CAND} candidates sharded x{n_gpus} (<= {per} each), one all_gather of 16-byte records for the argmax"
                        if n_gpus > 1 else "single GPU"),
        "l2": "inputs larger than L2 (factor 2.1 GB, K* / V 1.3 GB vs 126 MB L2); no explicit flush",
        "hyperparams": "reference defaults: log ell_d = 0, log sigma_f = 0, noise 0.01, UCB alpha 0.5, mean::Data",
        "seeds": {"data": 1234, "candidates": 1235},
    }


# --------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi during the timed region)
# --------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.lines: list[str] = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------
# CPU arm: the reference's own loops (oracle/_ref) or the oracle port, bounded sample, extrapolated
# --------------------------------------------------------------------------------------
_REF_LIB = None


def ref_lib():
    """oracle/_ref/libref_gp.so (the reference's gp.hpp / ucb.hpp compiled against the Eigen stand-in) or None."""
    global _REF_LIB
    if _REF_LIB is None:
        p = os.path.join(ROOT, "oracle", "_ref", "libref_gp.so")
        _REF_LIB = False
        if os.path.exists(p):
            try:
                lib = C.CDLL(p)
                vp, lg, i, d = C.c_void_p, C.c_long, C.c_int, C.c_double
                lib.ref_gp_bench.argtypes = [i, lg, i, vp, vp, d, lg, vp, i, vp, vp, vp, vp]
                lib.ref_gp_bench.restype = i
                _REF_LIB = lib
            except Exception:
                _REF_LIB = False
    return _REF_LIB or None


def cpu_kind() -> str:
    return "reference" if ref_lib() is not None else "port"


def cpu_sample(n_s: int, m_s: int, threads: int) -> dict:
    """One bounded sample: fit at N=n_s on one thread (Eigen's LLT is single-threaded in the reference) and m_s
    one-at-a-time UCB queries fanned over `threads` host threads (tools::par)."""
    from limbo_b200 import synth
    X = synth.points(1234, n_s, DIM)
    y = synth.targets(X)
    Xq = synth.points(1235, m_s, DIM)
    lib = ref_lib()
    if lib is not None:
        kid = {"SquaredExpARD": 0, "MaternFiveHalves": 1}[KERNEL_NAME]
        tf, tq, b, bi = C.c_double(), C.c_double(), C.c_double(), C.c_long()
        devnull = os.open(os.devnull, os.O_WRONLY)  # the reference's ~GP prints "'HPOpt' was never called!" on stdout
        saved = os.dup(1)
        sys.stdout.flush()
        os.dup2(devnull, 1)
        try:
            rc = lib.ref_gp_bench(kid, n_s, DIM, X.ctypes.data, y.ctypes.data, NOISE, m_s, Xq.ctypes.data, threads, C.addressof(tf),
                                  C.addressof(tq), C.addressof(b), C.addressof(bi))
        finally:
            os.dup2(saved, 1)
            os.close(saved)
            os.close(devnull)
        assert rc == 0, rc
        return {"t_fit": tf.value, "t_query": tq.value}
    from oracle import oracle as O
    g = O.OracleGP()
    g.set_data(X, (y - y.mean())[:, None])
    kid = {"SquaredExpARD": O.K_SE_ARD, "MaternFiveHalves": O.K_MATERN52}[KERNEL_NAME]
    g.set_kernel(kid, np.zeros(DIM + 1 if kid == O.K_SE_ARD else 2), NOISE)
    t0 = time.perf_counter()
    g.fit()
    t_fit = time.perf_counter() - t0
    t0 = time.perf_counter()
    mu, s2 = g.query(Xq, nthreads=threads)
    ucb = O.ucb(mu[:, 0] + y.mean(), s2, UCB_ALPHA)
    _ = int(np.argmax(ucb))
    t_q = time.perf_counter() - t0
    return {"t_fit": t_fit, "t_query": t_q}


def cpu_lapack_sample(n_s: int = 8192, m_s: int = 2048) -> dict | None:
    """NOT the reference's code path (which factors with single-threaded Eigen::LLT and predicts one point at a time): what a
    tuned host library does with the same mathematics - LAPACK dpotrf + ONE batched dtrsm over all candidates (scipy /
    OpenBLAS, all host cores).  Reported next to cpu_baseline so the GPU / CPU ratio can be read against a strong CPU too."""
    try:
        import scipy.linalg as sl
    except Exception:
        return None
    from limbo_b200 import synth
    X = synth.points(1234, n_s, DIM)
    y = synth.targets(X)
    Xq = synth.points(1235, m_s, DIM)
    if KERNEL_NAME != "SquaredExpARD":
        return None
    t0 = time.perf_counter()
    sq = (X ** 2).sum(1)
    K = np.exp(-0.5 * np.maximum(sq[:, None] + sq[None, :] - 2.0 * (X @ X.T), 0.0))
    K[np.diag_indices(n_s)] += NOISE + 1e-8
    t_k = time.perf_counter() - t0
    t0 = time.perf_counter()
    L = sl.cholesky(K, lower=True, overwrite_a=True, check_finite=False)
    alpha = sl.cho_solve((L, True), y - y.mean(), check_finite=False)
    t_fit = time.perf_counter() - t0
    t0 = time.perf_counter()
    sqq = (Xq ** 2).sum(1)
    Ks = np.exp(-0.5 * np.maximum(sq[:, None] + sqq[None, :] - 2.0 * (X @ Xq.T), 0.0))
    V = sl.solve_triangular(L, Ks, lower=True, check_finite=False)
    s2 = np.maximum(1.0 - (V ** 2).sum(0), 0.0) + NOISE
    ucb = Ks.T @ alpha + y.mean() + UCB_ALPHA * np.sqrt(s2)
    _ = int(np.argmax(ucb))
    t_q = time.perf_counter() - t0
    sec = t_k * (N_TRAIN / n_s) ** 2 + t_fit * (N_TRAIN / n_s) ** 3 + t_q * (M_CAND / m_s) * (N_TRAIN / n_s) ** 2
    return {"value": 1.0 / sec, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "host LAPACK, batched (not the reference's algorithm)",
            "sample": (f"numpy K build ({t_k:.2f} s) + scipy/OpenBLAS dpotrf ({t_fit:.2f} s) at N={n_s} + one dtrsm over {m_s} candidates "
                       f"({t_q:.2f} s), extrapolated to N={N_TRAIN}, M={M_CAND} by N^2 / N^3 / M*N^2 -> {sec:.1f} s per step")}


def cpu_step(n_s: int, m_s: int, threads: int) -> dict:
    """One bounded CPU step: the sample at n_s plus a half-size fit, so that the fit time is extrapolated with a fitted
    a N^2 + b N^3 model (the reference's fit is N^2/2 functor calls with heap temporaries - gp.hpp:552-562 - plus the N^3/3
    LLT; a pure N^3 law would overstate the CPU time) and the queries by M N^2."""
    full = cpu_sample(n_s, m_s, threads)
    if n_s >= N_TRAIN:
        sec_fit, model = full["t_fit"], "measured at full size"
    else:
        half = cpu_sample(n_s // 2, min(m_s, 2 * threads), threads)
        n1, n2, t1, t2 = float(n_s // 2), float(n_s), half["t_fit"], full["t_fit"]
        b = (t2 / n2 ** 2 - t1 / n1 ** 2) / (n2 - n1)
        a = t1 / n1 ** 2 - b * n1
        if a < 0 or b <= 0:  # noisy sample: fall back to the pure cubic law
            a, b = 0.0, t2 / n2 ** 3
        sec_fit = a * N_TRAIN ** 2 + b * N_TRAIN ** 3
        model = f"t_fit(N) = {a:.3e} N^2 + {b:.3e} N^3 fitted to N={n_s // 2} ({t1:.2f} s) and N={n_s} ({t2:.2f} s)"
    sec_q = full["t_query"] * (M_CAND / m_s) * (N_TRAIN / n_s) ** 2
    return {"t_fit": full["t_fit"], "t_query": full["t_query"], "sec_fit": sec_fit, "sec_query": sec_q, "sec": sec_fit + sec_q, "fit_model": model}


def pick_cpu_sample(budget_s: float, threads: int):
    """Largest sample (fit size n_s, m_s queries) whose cost (incl. the half-size fit) fits the per-step budget."""
    cal = cpu_sample(1024, 2 * threads, threads)
    m_s = max(256, 2 * threads)
    for n_s in (16384, 12288, 8192, 6144, 4096, 3072, 2048):
        if n_s > N_TRAIN:
            continue
        est = 1.125 * cal["t_fit"] * (n_s / 1024) ** 3 + cal["t_query"] * (m_s / (2 * threads)) * (n_s / 1024) ** 2
        if est <= budget_s:
            return n_s, m_s
    return 2048, m_s


def sample_text(kind: str, s: dict, n_s: int, m_s: int, threads: int) -> str:
    what = ("the reference's own gp.hpp / acqui/ucb.hpp loops (oracle/_ref/libref_gp.so: /root/reference headers over an Eigen stand-in with "
            "Eigen's blocked-LLT structure)" if kind == "reference" else "oracle port of the reference path")
    return (f"{what}: fit at N={n_s} on 1 thread like Eigen::LLT ({s['t_fit']:.2f} s) + {m_s} one-at-a-time UCB queries over {threads} threads "
            f"({s['t_query']:.2f} s); extrapolated to N={N_TRAIN}, M={M_CAND}: {s['fit_model']} -> {s['sec_fit']:.0f} s, queries by M*N^2 -> "
            f"{s['sec_query']:.0f} s; {s['sec']:.0f} s per step")


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    steps, warmup = args.steps, args.warmup
    kind = cpu_kind()
    # the timed steps should end within ~6 minutes: budget per step, sample size from a calibration run; warm-up steps use a
    # small sample (page-in, thread start-up) so that the budget goes to the largest fit that fits
    per_step = max(2.0, min(90.0, 360.0 / max(1, steps)))
    n_s, m_s = pick_cpu_sample(per_step, threads)
    for _ in range(warmup):
        cpu_sample(min(n_s, 1024), m_s, threads)
    samples = []
    t_all0 = time.perf_counter()
    for _ in range(steps):
        samples.append(cpu_step(n_s, m_s, threads))
    wall = time.perf_counter() - t_all0
    sec = float(np.mean([s["sec"] for s in samples]))
    value = 1.0 / sec
    med = sorted(samples, key=lambda s: s["sec"])[len(samples) // 2]
    sample = sample_text(kind, med, n_s, m_s, threads) + f" (median step shown; measured {wall / max(1, steps):.2f} s of CPU work per step)"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": DATA, "config": workload_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": ("the same GLOBAL job at every --gpus N (the GPU arm strong-scales it); the CPU path has no device, so its value "
                 "does not depend on N"),
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------
PC = ["kbuild", "potf2", "trsm_panel", "syrk", "syrk_col", "trsv", "kstar", "qstep", "qreduce", "acq", "trtri", "lauum", "grad", "other"]


def syrk_flops_per_fit(n: int) -> float:
    """Algorithmic flops of the main-stream trailing updates (profile class "syrk") of one factorisation: panels are taken in
    quads (k .. k+3); the update of the matrix right of the quad has order m = (T - k - 4) * 128 and costs m (m + 1) * 512 flops
    (lower triangle incl. diagonal, 2 flops per MAC, K = 512).  (LB_POTRF_QUAD=0, the pair scheme of round 1: K = 256.)"""
    nb, tot = 128, 0.0
    t = (n + nb - 1) // nb
    quad = os.environ.get("LB_POTRF_QUAD", "1") != "0"
    g = 4 if quad else 2
    for k in range(0, t, g):
        m = max(0, (t - k - g)) * nb
        tot += float(m) * (m + 1) * (g * nb)
    return tot


def fp64_tensor_peak() -> tuple[float, str]:
    p = os.path.join(ROOT, "profiles", "fp64_peaks.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return float(j["dmma_tflops"]), f"builder-measured DMMA peak ({j.get('source', 'tools/microbench.cu')}); MEASURED_PEAKS.json has no fp64 figure"
        except Exception:
            pass
    return 40.0, "nominal B200 fp64 tensor peak (40 TFLOP/s); MEASURED_PEAKS.json has no fp64 figure"


def measured_peaks() -> dict:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return json.load(open(p))
    except Exception:
        return {}


def ncu_traffic(kernel: str):
    """DRAM bytes of one captured launch (ncu --set full), from the committed profile summaries (latest round first)."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            j = json.load(open(os.path.join(ROOT, "profiles", name)))[kernel]
            j = dict(j)
            j["source"] = "profiles/" + name
            return j["dram_bytes"], j
        except Exception:
            continue
    return None, None


def hbm_peak() -> tuple[float, str]:
    mp = measured_peaks()
    if "hbm_gbs" in mp:
        return float(mp["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def prof_api(lib):
    lib.lb_profile_enable.argtypes = [C.c_void_p, C.c_int]
    lib.lb_profile_read.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]


def prof_read(lib, h) -> dict:
    ms = (C.c_double * len(PC))()
    cnt = (C.c_longlong * len(PC))()
    lib.lb_profile_read(h, ms, cnt, 1)
    return {PC[i]: {"ms_total": ms[i], "launches": int(cnt[i])} for i in range(len(PC)) if cnt[i]}


def roofline_table(prof: dict, steps: int, t_ms: float, n: int, d: int, m_local: int) -> list[dict]:
    """One row per profiled kernel class: algorithmic work per launch (DESIGN.md §4) / average launch time, against the
    roofline that bounds it.  m_local = candidates this GPU scores per step."""
    peak_t, peak_t_src = fp64_tensor_peak()
    peak_h, peak_h_src = hbm_peak()
    rows = []

    def add(cls, kernel, bound, work_per_step, unit_scale, peak, src, note=None):
        if cls not in prof or not prof[cls]["launches"]:
            return
        tot_ms, launches = prof[cls]["ms_total"], prof[cls]["launches"]
        per_launch = work_per_step * steps / launches
        avg_ms = tot_ms / launches
        ach = per_launch / (avg_ms * 1e-3) / unit_scale
        row = {"kernel": kernel, "class": cls, "bound": bound, "achieved": ach, "peak": peak, "unit": "TFLOP/s" if bound == "tensor" else "GB/s",
               "frac": ach / peak, "share_of_step": tot_ms / t_ms, "avg_launch_ms": avg_ms, "launches_per_step": launches / steps,
               ("algorithmic_flops_per_launch" if bound == "tensor" else "algorithmic_bytes_per_launch"): per_launch, "peak_source": src}
        if note:
            row["note"] = note
        rows.append(row)

    qname = ("panel_update_kernel + panel_solve_kernel (V = L^-1 K* over 2048-row super-blocks, fp64 DMMA)" if m_local >= 256
             else "query_slab_kernel (fused K* + blocked TRSM + mu / sigma^2, fp64 DMMA)")
    add("qstep", qname, "tensor", float(m_local) * n * n, 1e12, peak_t, peak_t_src,
        "M N^2 flops per batch (triangular solve, 2 flops per MAC on N^2 / 2); launches of one batch are averaged")
    add("kstar", "kstar_kernel (K* = k(X, Xq), N x M)", "hbm", 8.0 * n * m_local + 8.0 * (n + m_local) * d, 1e9, peak_h, peak_h_src)
    add("syrk", "syrk_kernel K=512 (Cholesky trailing update in panel quads, fp64 DMMA)", "tensor", syrk_flops_per_fit(n), 1e12, peak_t, peak_t_src)
    add("kbuild", "kbuild_kernel (N x N kernel matrix)", "hbm", 8.0 * n * n + 8.0 * n * d, 1e9, peak_h, peak_h_src)
    add("trsv", "trsv_fwd/bwd_kernel (alpha = L^-T L^-1 obs_mean)", "hbm", 2 * 4.0 * n * n, 1e9, peak_h, peak_h_src,
        "4 N^2 bytes per direction (lower triangle of L read once)")
    add("potf2", "potf2_inv_kernel (128 x 128 diagonal block + inverse)", "tensor", (n / 128) * (128 ** 3 / 3 + 2 * 128 ** 3 / 3), 1e12, peak_t,
        peak_t_src, "latency bound (128-pivot chain), side stream, hidden by look-ahead")
    add("trsm_panel", "trsm_panel_kernel (panel solve)", "tensor", sum(2.0 * 128 ** 3 * (n // 128 - k - 1) for k in range(n // 128)), 1e12, peak_t,
        peak_t_src, "side stream, runs under the trailing update")
    tt = n // 128
    quad = os.environ.get("LB_POTRF_QUAD", "1") != "0"
    col_flops = sum(2.0 * 128 ** 3 * (tt - k - 1) for k in range(0, tt, 2))  # block column k+1 updated with panel k (K = 128)
    if quad:  # inside a quad: block columns k+2, k+3 updated with the pair (k, k+1), K = 256
        for k in range(0, tt, 4):
            for j in (k + 2, k + 3):
                if j < tt:
                    col_flops += 2.0 * 128 * 128 * 256 * (tt - j)
    add("syrk_col", "syrk_kernel K=128 / K=256 (look-ahead column updates inside a panel quad)", "tensor", col_flops, 1e12,
        peak_t, peak_t_src, "side stream")
    rows.sort(key=lambda r: -r["share_of_step"])
    return rows


DUMP_SEED, DUMP_L_ROWS = 2024, 256


def dump_outputs(out_dir: str, lib, h, n: int, best: tuple[float, int]) -> None:
    """--dump-outputs: what the last timed step hands its caller, as float64 .npy files, so that two builds can be compared
    output for output: the UCB argmax (value, global index), alpha (N) and a fixed, seeded sample of DUMP_L_ROWS rows of the
    Cholesky factor L (the whole factor is 2.1 GB at N=16384; the sample is 32 MB)."""
    from limbo_b200 import _lib
    L = np.empty((n, n), order="F")
    _lib.check(lib.lb_get(h, _lib.GET_L, L.ctypes.data), "lb_get L")
    alpha = np.empty(n)
    _lib.check(lib.lb_get(h, _lib.GET_ALPHA, alpha.ctypes.data), "lb_get alpha")
    rows = np.sort(np.random.default_rng(DUMP_SEED).choice(n, min(n, DUMP_L_ROWS), replace=False))
    out = {"ucb_best_value": np.array([best[0]]), "ucb_best_index": np.array([best[1]], dtype=np.float64), "alpha": alpha,
           "L_rows": np.ascontiguousarray(L[rows]), "L_row_index": rows.astype(np.float64)}
    del L
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_config4(args, torch, dist, dev, rank, world, lib, precision: str = "tf32", m_total: int = 1_000_000, steps: int = 2) -> dict | None:
    """BASELINE.json config 4: N=16384, D=12, reduced-precision scoring, 1M EI candidates sharded over the ranks, one
    all_gather for the argmax.  The timed step includes the fp64 fit, the inversion of the factor and its cast (replicated on
    every rank), the f_max scan, and the sharded scoring + collective."""
    from limbo_b200 import _lib, acqui, kernel, mean, model, synth
    from limbo_b200 import dist as lbd
    n, d = 16384, 12
    X = synth.points(1234, n, d)
    y = synth.targets(X)
    lo, hi = lbd.shard_range(m_total, rank, world)
    Xq = synth.points(4321, m_total, d)[lo:hi]
    gp = model.GP(d, 1, kernel=kernel.SquaredExpARD, mean=mean.Data, device=dev.index, precision=precision)
    st = torch.cuda.current_stream(dev)
    gp.set_stream(st.cuda_stream)
    dXq = torch.from_numpy(np.ascontiguousarray(Xq)).to(dev)
    dBest = torch.zeros(1, dtype=torch.float64, device=dev)
    dIdx = torch.zeros(1, dtype=torch.int64, device=dev)
    m_loc = hi - lo
    mean_const = float(y.mean())
    ei = acqui.EI(gp)
    ap = np.array([0.0, 0.0])  # EI parameters: f_max (refreshed per fit), jitter 0
    out = {}

    fitter = None
    if world > 1 and not args.replicated_fit:  # the fp64 fit is the distributed one (dist_fit.py)
        from limbo_b200 import dist_fit
        gp.compute(X, y[:, None], compute_kernel=False)
        fitter = dist_fit.DistFit(gp, rank, world, dev)
        if not fitter.supported(gp):
            fitter.close()
            fitter = None

    dinv = None
    if world > 1 and not args.replicated_inverse:  # every rank inverts its column tiles of the factor, one all_gather (dist_inv.py)
        from limbo_b200 import dist_inv
        dinv = dist_inv.DistInverse(gp, rank, world, dev)

    def step():
        if fitter is not None:
            gp.compute(X, y[:, None], compute_kernel=False)
            fitter.fit(gp)
        else:
            gp.compute(X, y[:, None])                      # fp64 fit through the public API (H2D inside)
        if dinv is not None:
            dinv.prepare(gp)
        ei._nb_samples = -1
        ei._update_f_max(acqui.first_elem)                 # ei.hpp:100-108: f_max = max_i mu(x_i), one batched pass over the N samples
        ap[0] = ei._f_max
        _lib.check(lib.lb_acq_argmax_dev(gp._h, 1, ap.ctypes.data, m_loc, dXq.data_ptr(), None, mean_const, None, dBest.data_ptr(),
                                         dIdx.data_ptr()), "acq_argmax_dev")
        _lib.check(lib.lb_sync(gp._h), "lb_sync")
        return lbd.allgather_argmax(float(dBest.item()), int(dIdx.item()) + lo, device=dev)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    step()  # warm-up: allocations, kernel attributes
    sync_all()
    lib.lb_profile_enable(gp._h, 1)
    prof_read(lib, gp._h)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record(st)
    for _ in range(steps):
        best = step()
    e1.record(st)
    sync_all()
    ms = max(e0.elapsed_time(e1), 0.0) / steps
    prof = prof_read(lib, gp._h)
    lib.lb_profile_enable(gp._h, 0)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    stage = {k: v["ms_total"] / steps for k, v in prof.items()}
    fit_ms = sum(stage.get(k, 0.0) for k in ("kbuild", "syrk", "trsv")) + 0.0
    if fitter is not None:
        # the distributed fit runs on the fitter's own handle / streams (not in this handle's stage clocks): one extra fit, wall-timed
        # between full synchronisations on every rank
        sync_all()
        tf = time.perf_counter()
        gp.compute(X, y[:, None], compute_kernel=False)
        fitter.fit(gp)
        _lib.check(lib.lb_sync(gp._h), "lb_sync")
        torch.cuda.synchronize(dev)
        fit_ms = (time.perf_counter() - tf) * 1e3
        sync_all()
        fitter.close()
    if dinv is not None:
        dinv.close()
    inv_ms = stage.get("trtri", 0.0) + stage.get("other", 0.0)
    score_ms = stage.get("kstar", 0.0) + stage.get("qstep", 0.0) + stage.get("qreduce", 0.0)
    mp = measured_peaks()
    # the GEMM is timed alone (CUDA events around its launches): burst figure; tf32 runs at half the 16-bit rate
    bf16 = float(mp.get("bf16_tflops", 1676.8))
    tens_peak = bf16 / 2 if precision == "tf32" else bf16
    flops = float(m_loc) * n * n * (3.0 if precision == "fp16x3" else 1.0)  # split operands: three products per MAC
    gemm_ms = stage.get("qstep", 0.0)
    out = {
        "workload": f"config 4: N={n}, D={d}, SquaredExpARD, fp64 fit + {precision} scoring of {m_total} EI candidates, sharded x{world}",
        "metric": "EI candidates/s (fit + L^-1 + cast inside the timed step)", "value": m_total / (ms * 1e-3), "unit": "candidates/s",
        "ms_per_step": ms, "n_gpus": world, "steps": steps, "scaling": "strong", "precision": precision,
        "stage_ms_rank0": stage, "fit_ms_rank0": fit_ms, "invert_and_cast_ms_rank0": inv_ms, "score_ms_rank0": score_ms,
        "scoring_only_candidates_per_s": m_total / (score_ms * 1e-3) if score_ms > 0 else None,
        "fit_scheme": "distributed (dist_fit.py)" if fitter is not None else ("replicated" if world > 1 else "single GPU"),
        "inverse_scheme": "column tiles per rank + one all_gather (dist_inv.py)" if dinv is not None else ("replicated" if world > 1 else "single GPU"),
        "limiter": ((f"distributed fp64 fit {fit_ms:.0f} ms (wall-timed on rank 0 in one extra step; its serial panel chain) + inversion by column "
                     f"tiles, cast and all_gather ({inv_ms:.0f} ms of kernels on rank 0) + {score_ms:.0f} ms of sharded scoring") if (fitter is not None and dinv is not None) else
                    (f"inversion of the factor + cast ({inv_ms:.0f} ms) are replicated on every rank (every rank scores against all of L^-1); the "
                     f"fp64 fit is distributed ({fit_ms:.0f} ms, wall-timed on rank 0 in one extra step), the {score_ms:.0f} ms of scoring shard") if fitter is not None else
                    (f"fp64 fit ({fit_ms:.0f} ms) + inversion/cast ({inv_ms:.0f} ms) are replicated on every rank (Amdahl); only the "
                     f"{score_ms:.0f} ms of scoring shard")),
        "best": {"value": best[0], "index": best[1]},
        "roofline": {"kernel": ("pair_split_gemm_norm_kernel" if precision == "fp16x3" else "pair_gemm_norm_kernel") + " (tcgen05 cta_group::2, sigma^2 GEMM)", "bound": "tensor",
                     "achieved": flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else None, "peak": tens_peak, "unit": "TFLOP/s",
                     "frac": (flops / (gemm_ms * 1e-3) / 1e12 / tens_peak) if gemm_ms > 0 else None,
                     "algorithmic_flops_per_step": flops,
                     "peak_source": ("MEASURED_PEAKS.json bf16_tflops (cuBLAS bf16 burst; fp16 MMAs run at the same rate)"
                                     + (" / 2 (tf32 runs at half the 16-bit rate)" if precision == "tf32" else ""))},
    }
    del gp
    return out


def run_config5(args, torch, dist, dev, rank, world, n: int = 65536) -> dict | None:
    """BASELINE.json config 5: right-looking block Cholesky of the N=65536 kernel matrix, 1-D block-cyclic 256-column panels
    over the ranks, one panel broadcast per step (limbo_b200/dist_chol.py).  One timed factorisation after a small warm-up."""
    from limbo_b200 import dist_chol, kernel, synth
    free, _total = torch.cuda.mem_get_info(dev)
    need = 8.0 * n * n / world + 2 * 8.0 * 256 * n + (2 << 30)
    if free < need:
        return {"skipped": f"needs {need / 1e9:.0f} GB per GPU at {world} GPU(s), {free / 1e9:.0f} GB free"}
    d = 6
    kf = kernel.SquaredExpARD(None, d)
    kf.set_h_params(np.concatenate([np.full(d, np.log(0.3)), [0.0]]))
    # warm-up at a small order: NCCL communicator, kernel attributes, allocator
    w = dist_chol.DistCholesky(synth.points(1234, 4096, d), kf, rank, world, dev)
    w.build(); w.factor(); w.close()
    del w
    X = synth.points(1234, n, d)
    dc = dist_chol.DistCholesky(X, kf, rank, world, dev)
    dc.build()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(dc.main)
    info, logdet = dc.factor()
    e1.record(dc.main)
    torch.cuda.synchronize(dev)
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    # || L (L^T v) - K v || / || K v || with K regenerated from X
    g = torch.Generator(device="cpu").manual_seed(7)
    v = torch.randn(dc.Nd, generator=g, dtype=torch.float64).to(dev)
    cols = torch.from_numpy(dc.global_columns()).to(dev)
    with torch.cuda.stream(dc.main):
        wv = dc.L.T @ (dc.L @ v)
        dc.build()
        kv = dc.L.T @ v[cols]
    dc.main.synchronize()
    if world > 1:
        dist.all_reduce(wv)
        dist.all_reduce(kv)
    resid = float(((wv - kv).norm() / kv.norm()).item())
    peak_t, peak_src = fp64_tensor_peak()
    tf = n ** 3 / 3 / (ms * 1e-3) / 1e12
    out = {"workload": f"config 5: N={n}, D={d}, SquaredExpARD fp64 Cholesky, 1-D block-cyclic 256-column panels over {world} GPU(s), panel broadcast per step",
           "metric": "factorisations/s", "value": 1e3 / ms, "unit": "1/s", "ms": ms, "n_gpus": world, "scaling": "strong",
           "tflops_total": tf, "tflops_per_gpu": tf / world, "frac_of_dmma_peak_per_gpu": tf / world / peak_t, "peak_source": peak_src,
           "info": info, "logdet": logdet, "matvec_rel_residual": resid, "local_gb": dc.L.numel() * 8 / 1e9, "launches_rank0": dc.launches,
           "limiter": ("owner's serial panel chain (potf2 -> trsm -> column update -> potf2 -> trsm -> pack) + one panel broadcast per "
                       "256 columns on the critical path once the per-GPU trailing update is shorter than that chain" if world > 1 else "single GPU")}
    dc.close()
    del dc
    torch.cuda.empty_cache()
    return out


def run_ours(args) -> None:
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (limbo_b200 has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from limbo_b200 import _lib, acqui, kernel, mean, model, synth
    from limbo_b200 import dist as lbdist

    lib = _lib.load()
    prof_api(lib)

    steps, warmup = args.steps, max(args.warmup, 3)
    n, d, m = N_TRAIN, DIM, M_CAND
    X = synth.points(1234, n, d)
    y = synth.targets(X)
    Xq_all = synth.points(1235, m, d)          # the global candidate batch (same on every rank)
    lo, hi = lbdist.shard_range(m, rank, world)
    Xq = np.ascontiguousarray(Xq_all[lo:hi])   # this rank's contiguous shard
    m_loc = hi - lo

    kcls = getattr(kernel, KERNEL_NAME)
    kid_dev = kcls.kernel_id
    gp = model.GP(d, 1, kernel=kcls, mean=mean.Data, device=local_rank)
    h = gp._h
    # a real (non-default) stream: the library and the timing events must share it
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    gp.set_stream(stream.cuda_stream)
    # N > 1: the fit itself is distributed over the ranks (limbo_b200/dist_fit.py) unless --replicated-fit
    fitter = None
    if world > 1 and not args.replicated_fit:
        from limbo_b200 import dist_fit
        gp.compute(X, y[:, None], compute_kernel=False)  # host-side state of the model (samples, obs_mean); no device fit
        fitter = dist_fit.DistFit(gp, rank, world, dev)
        if not fitter.supported(gp):
            fitter.close()
            fitter = None

    # ---------------- device-resident leg ("value") ----------------
    dX = torch.from_numpy(X).to(dev)
    om = (y - y.mean())
    dY = torch.from_numpy(om).to(dev)
    dXq = torch.from_numpy(Xq).to(dev)
    dBest = torch.zeros(1, dtype=torch.float64, device=dev)
    dIdx = torch.zeros(1, dtype=torch.int64, device=dev)
    ap = np.array([UCB_ALPHA, 0.0])
    hp = np.zeros(d + 1 if KERNEL_NAME == "SquaredExpARD" else 2)
    mean_const = float(y.mean())
    gather_buf = [torch.zeros(2, dtype=torch.float64, device=dev) for _ in range(world)] if world > 1 else None

    def step_dev():
        _lib.check(lib.lb_set_data_dev(h, n, d, 1, dX.data_ptr(), dY.data_ptr()), "set_data_dev")
        _lib.check(lib.lb_set_kernel(h, kid_dev, hp.ctypes.data, hp.size, NOISE), "set_kernel")
        if fitter is not None:
            torch.cuda.synchronize(dev)  # so that the wall clock below times the fit alone (fit() returns synchronised anyway)
            t_f = time.perf_counter()
            fitter.fit(gp, push=False)  # distributed K -> L (assembled on every rank) -> alpha; returns synchronised
            fit_wall.append((time.perf_counter() - t_f) * 1e3)
        else:
            _lib.check(lib.lb_fit_async(h), "fit_async")
        _lib.check(lib.lb_acq_argmax_dev(h, 0, ap.ctypes.data, m_loc, dXq.data_ptr(), None, mean_const, None, dBest.data_ptr(),
                                         dIdx.data_ptr()), "acq_argmax_dev")
        if world > 1:  # one collective: (value, global index) records, reduced locally
            rec = torch.stack([dBest[0], (dIdx[0] + lo).to(torch.float64)])
            dist.all_gather(gather_buf, rec)

    fit_wall: list[float] = []

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    for _ in range(warmup):
        step_dev()
    sync_all()
    _lib.check(lib.lb_check_info(h), "cholesky info")
    fit_wall.clear()

    lib.lb_profile_enable(h, 1)
    prof_read(lib, h)
    if fitter is not None:
        lib.lb_profile_enable(fitter._h_main, 1)
        prof_read(lib, fitter._h_main)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = gp.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record(stream)
    for _ in range(steps):
        step_dev()
    e1.record(stream)
    sync_all()
    t_ms = e0.elapsed_time(e1)
    launches = gp.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    prof = prof_read(lib, h)
    lib.lb_profile_enable(h, 0)
    if fitter is not None:  # the trailing updates of the distributed fit run on the fitter's own handle
        for k, v in prof_read(lib, fitter._h_main).items():
            if k in prof:
                prof[k]["ms_total"] += v["ms_total"]; prof[k]["launches"] += v["launches"]
            else:
                prof[k] = v
        lib.lb_profile_enable(fitter._h_main, 0)
    fit_wall_ms = float(np.mean(fit_wall)) if fit_wall else None
    tt = torch.tensor([t_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_ms = float(tt.item())
    ms_per_step = t_ms / steps
    value = 1.0 / (ms_per_step * 1e-3)  # global jobs per second (one job = fit + all M candidates), whatever the GPU count
    if args.dump_outputs and rank == 0:
        if world > 1:
            recs = torch.stack(gather_buf).cpu().numpy()
            best = lbdist.reduce_records(recs[:, 0], recs[:, 1].astype(np.int64))
        else:
            best = (float(dBest.item()), int(dIdx.item()))
        dump_outputs(args.dump_outputs, lib, h, n, best)

    # ---------------- end-to-end leg through the public host API ----------------
    gp2 = model.GP(d, 1, kernel=kcls, mean=mean.Data, device=local_rank)
    gp2.set_stream(stream.cuda_stream)
    Xp = torch.from_numpy(X).pin_memory()
    yp = torch.from_numpy(y[:, None].copy()).pin_memory()
    Xqp = torch.from_numpy(Xq_all).pin_memory()
    Xl, yl, Xql = Xp.numpy(), yp.numpy(), Xqp.numpy()  # pinned host buffers, one point per row
    ucb = acqui.UCB(gp2)
    fitter2 = None
    if fitter is not None:
        gp2.compute(Xl, yl, compute_kernel=False)
        fitter2 = dist_fit.DistFit(gp2, rank, world, dev)

    def step_e2e():
        if fitter2 is not None:
            gp2.compute(Xl, yl, compute_kernel=False)  # host-side model state; the device fit is the distributed one
            fitter2.fit(gp2)                           # H2D of samples / obs_mean inside
        else:
            gp2.compute(Xl, yl)                 # host samples/observations in, H2D inside
        # host candidates in, (value, global index) out; N > 1: this rank's shard + the one collective
        return lbdist.sharded_acq_argmax(ucb, Xql, rank, world, device=dev)

    e2e_steps = max(2, min(steps, 5))
    step_e2e()
    sync_all()
    t0 = time.perf_counter()
    e0.record(stream)
    for _ in range(e2e_steps):
        best_e2e = step_e2e()
    e1.record(stream)
    sync_all()
    t_e2e_ms = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
    tt = torch.tensor([t_e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    e2e_value = 1.0 / (float(tt.item()) / e2e_steps * 1e-3)
    # the other kernel north_star names for the K build (MaternFiveHalves), timed alone at the same N: driver-visible roofline
    roof_km = None
    if rank == 0 and args.workload == "n16384_se_ard":
        try:
            gm = model.GP(d, 1, kernel=kernel.MaternFiveHalves, mean=mean.Data, device=local_rank)
            gm.set_stream(stream.cuda_stream)
            hm = np.zeros(2)
            _lib.check(lib.lb_set_data_dev(gm._h, n, d, 1, dX.data_ptr(), dY.data_ptr()), "set_data_dev")
            _lib.check(lib.lb_set_kernel(gm._h, kernel.MaternFiveHalves.kernel_id, hm.ctypes.data, hm.size, NOISE), "set_kernel")
            lib.lb_stage_kbuild.argtypes = [C.c_void_p]
            for _ in range(3):
                _lib.check(lib.lb_stage_kbuild(gm._h), "stage_kbuild")
            ek0, ek1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(dev)
            ek0.record(stream)
            for _ in range(10):
                _lib.check(lib.lb_stage_kbuild(gm._h), "stage_kbuild")
            ek1.record(stream)
            torch.cuda.synchronize(dev)
            km_ms = ek0.elapsed_time(ek1) / 10
            peak_h, peak_h_src = hbm_peak()
            byts = 8.0 * n * n + 8.0 * n * d
            roof_km = {"kernel": "kbuild_kernel<MaternFiveHalves> (N x N kernel matrix; includes the tiny scale_x launch)", "bound": "hbm",
                       "achieved": byts / (km_ms * 1e-3) / 1e9, "peak": peak_h, "unit": "GB/s", "frac": byts / (km_ms * 1e-3) / 1e9 / peak_h,
                       "avg_launch_ms": km_ms, "algorithmic_bytes_per_launch": byts, "peak_source": peak_h_src,
                       "traffic": (ncu_traffic("kbuild_kernel_matern52")[0])}
            del gm
        except Exception as e:
            roof_km = {"error": repr(e)}
    h2d = n * d * 8 + n * 8 + m_loc * d * 8 + 2 * 8
    d2h = 8 + 8 + 8
    if fitter2 is not None:
        fitter2.close()
    del gp2
    if fitter is not None:
        fitter.close()

    if rank == 0:
        stage = {k: v["ms_total"] / steps for k, v in prof.items()}
        table = roofline_table(prof, steps, t_ms, n, d, m_loc)
        roof = {}
        if table:
            top = dict(table[0])
            cls = top["class"]
            kname = {"qstep": ("panel_update_kernel" if m_loc >= 256 else "query_slab_kernel"), "syrk": "syrk_kernel", "kbuild": "kbuild_kernel"}.get(cls)
            tr, cap = ncu_traffic(kname) if kname else (None, None)
            top["traffic"] = tr
            top["traffic_capture"] = cap
            roof = top
        roof_k = next((dict(r) for r in table if r["class"] == "kbuild"), {})
        if roof_k:
            roof_k["traffic"] = ncu_traffic("kbuild_kernel")[0]
        fit_ms = sum(stage.get(k, 0.0) for k in ("kbuild", "syrk", "trsv"))
        q_ms = stage.get("qstep", 0.0)
        # CPU baseline on a bounded sample (rank 0, N=1 only)
        cpu = None
        if world == 1 and not args.no_cpu:
            threads = os.cpu_count() or 1
            n_s, m_s = pick_cpu_sample(55.0, threads)
            s = cpu_step(n_s, m_s, threads)
            cpu = {"value": 1.0 / s["sec"], "unit": UNIT, "cores": threads, "kind": cpu_kind(), "sample": sample_text(cpu_kind(), s, n_s, m_s, threads)}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": DATA, "config": workload_config(world), "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                    "api": "limbo_b200.model.GP.compute + limbo_b200.dist.sharded_acq_argmax(acqui.UCB) (pinned host buffers)",
                    "best": {"value": best_e2e[0], "index": best_e2e[1]}},
            "gpu_launches": int(launches), "roofline": roof, "roofline_kbuild": roof_k, "roofline_kbuild_matern52": roof_km, "roofline_kernels": table,
            "cpu_baseline": cpu,
            "cpu_lapack_batched": (cpu_lapack_sample() if (world == 1 and not args.no_cpu) else None),
            "stage_ms_per_step": stage,
            "fit": ({"scheme": "distributed (limbo_b200/dist_fit.py)", "wall_ms_per_fit_rank0": fit_wall_ms} if (world > 1 and fit_wall_ms is not None)
                    else {"scheme": "replicated on every rank" if world > 1 else "single GPU"}),
            "limiter": ((f"strong scaling of one global job: distributed fit {fit_wall_ms:.1f} ms (trailing update {stage.get('syrk', 0.0):.1f} ms per GPU; the rest is the "
                         f"owner's serial panel chain potf2 -> trsm -> column update -> potf2 -> trsm -> pack + one broadcast per 256 columns, exposed once "
                         f"the per-GPU update is shorter than the chain) + sharded query {q_ms:.1f} ms ({m_loc} of {m} candidates)") if (world > 1 and fit_wall_ms is not None)
                        else (f"strong scaling of one global job: the fit ({fit_ms:.1f} ms of main-stream kernels per step) is replicated on every "
                              f"rank and does not shrink with N; only the query ({q_ms:.1f} ms here for {m_loc} of {m} candidates) shards") if world > 1
                        else "single GPU: fp64 datapath (panel_update / panel_solve + syrk_kernel, all DMMA)"),
        }
    else:
        line = None

    # ---------------- sub-records: the multi-GPU splits BASELINE.json names ----------------
    # Safety net: the headline is measured; whatever happens in a sub-record (a collective that never returns cannot be caught
    # as an exception) must not cost the line.  Every rank arms the same deadline; when it fires, rank 0 prints the line with
    # the sub-records gathered so far and every rank leaves.
    sub = {"config4": None, "config4_fp16": None, "config4_fp16x3": None, "config5": None}

    def emit():
        if rank == 0:
            print(json.dumps({**line, **sub}))
            sys.stdout.flush()

    def watchdog():
        for k, v in sub.items():
            if v is None:
                sub[k] = {"error": f"sub-record did not finish within {args.sub_timeout} s"}
        emit()
        os._exit(0)

    if not args.no_sub and args.workload == "n16384_se_ard":
        timer = threading.Timer(float(args.sub_timeout), watchdog)
        timer.daemon = True
        timer.start()
        try:
            sub["config4"] = run_config4(args, torch, dist, dev, rank, world, lib, "tf32")
            sub["config4_fp16"] = run_config4(args, torch, dist, dev, rank, world, lib, "fp16")
            sub["config4_fp16x3"] = run_config4(args, torch, dist, dev, rank, world, lib, "fp16x3", steps=1)
        except Exception as e:  # a sub-record must never take the headline down
            sub["config4"] = sub["config4"] or {"error": repr(e)}
        try:
            lib.lb_pool_trim()
            torch.cuda.empty_cache()
            sub["config5"] = run_config5(args, torch, dist, dev, rank, world)
        except Exception as e:
            sub["config5"] = {"error": repr(e)}
        timer.cancel()
    emit()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_config4_workload(args) -> None:
    """--workload config4: the config-4 step as the headline line of this run (own metric)."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); lr = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(lr)
    dev = torch.device("cuda", lr)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from limbo_b200 import _lib
    lib = _lib.load()
    prof_api(lib)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    sampler = ClockSampler(lr)
    if rank == 0:
        sampler.start()
    rec = run_config4(args, torch, dist, dev, rank, world, lib, args.precision, steps=max(1, args.steps))
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        line = {"metric": "EI candidates/s at N=16384,D=12 (fp64 fit + reduced-precision scoring of 1M candidates + argmax)",
                "value": rec["value"], "unit": rec["unit"], "n_gpus": world, "steps": rec["steps"], "warmup": 1, "ms_per_step": rec["ms_per_step"],
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": args.precision, "data": DATA,
                "config": {"workload": rec["workload"]}, "clocks": clocks, "roofline": rec["roofline"], "detail": rec}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline sample")
    ap.add_argument("--no-sub", action="store_true", help="skip the config4 / config5 sub-records")
    ap.add_argument("--sub-timeout", type=int, default=240, help="seconds after which the line is printed without the unfinished sub-records")
    ap.add_argument("--replicated-fit", action="store_true", help="N > 1: every rank refits alone (round-1 scheme) instead of the distributed fit")
    ap.add_argument("--replicated-inverse", action="store_true",
                    help="N > 1, config 4: every rank inverts the whole factor (round-1 scheme) instead of its column tiles + one all_gather")
    ap.add_argument("--workload", default="n16384_se_ard", choices=sorted(WORKLOADS) + ["config4"])
    ap.add_argument("--precision", default="tf32", choices=["tf32", "fp16"], help="--workload config4 only")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.workload == "config4"):
        ap.error("--dump-outputs applies to the fit + UCB workloads of --impl ours")
    if args.workload == "config4":
        if args.impl == "reference":
            print(json.dumps({"impl": "reference", "unavailable": "config 4 is a reduced-precision GPU workload; the reference arm is defined for the headline workload"}))
            return
        run_config4_workload(args)
        return
    global N_TRAIN, DIM, M_CAND, KERNEL_NAME, METRIC
    N_TRAIN, DIM, M_CAND, KERNEL_NAME = WORKLOADS[args.workload]
    if args.workload != "n16384_se_ard":
        METRIC = f"GP fit+query/s at N={N_TRAIN},D={DIM} ({KERNEL_NAME}; fit = K-build+Cholesky+alpha, query = {M_CAND} UCB candidates+argmax, fp64)"
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
