#!/usr/bin/env python
"""BatchBQ(kernel=PeriodicKernel): P problems over an angle, each a von Mises likelihood with its own mean and concentration
(the reference's tests/util.py likelihood), advanced in lock-step.  One JSON line per case on stdout:

    python bench_batch_periodic.py > profiles/batch_periodic_r06.jsonl

Every problem starts at ns = 16 observations spread over [-pi, pi), with the 1000-point angle grid of BQ._approx and a
1000-point query grid over the same range.  Reported:
  * 20 rounds of choose_next (fixed hyper-parameters) + add_observations, in host mode and in device-resident mode: wall
    time of all rounds (each round ends in a device synchronise: the chosen points come back to the host);
  * one batched value-and-gradient evaluation of all P problems (BatchBQ.log_lh_grad with "h", "w", "p") next to one
    BatchBQ.log_lh call (two setups of the batch: the proposal and the restore); each shape is run once before it is timed;
  * the whole fit_hypers(["h", "w", "p"]) from the start: wall time, iterations, evaluations, converged problems and the
    median gain of log_lh;
  * for context, the same 20 rounds done by a loop of BQ objects over the first --loop problems (expected_squared_mean over
    the grid, its first maximiser, add_observation), extrapolated linearly to P."""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
warnings.simplefilter("ignore")

PARAMS = ["h", "w", "p"]
PARAMS_TL, PARAMS_L = (3.0, 0.6, 1.0, 0.1), (0.3, 0.5, 1.0, 1e-3)     # (h, w, p, s); noise so that the fit is bounded
OPT = dict(n_candidate=10, candidate_thresh=0.05, x_mean=0.0, x_var=10.0)
NS0, ROUNDS, NA = 16, 20, 1000


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except Exception:
        import torch
        return torch.cuda.get_device_name(0), "unknown"


def spread(v):
    v = np.asarray(v, dtype=np.float64)
    return {"min": round(float(v.min()), 4), "median": round(float(np.median(v)), 4), "max": round(float(v.max()), 4), "n": int(v.size)}


def likelihoods(P):
    from scipy.special import iv
    rs = np.random.RandomState(0)
    mu, kappa = rs.uniform(-np.pi, np.pi, P), rs.uniform(0.5, 3.0, P)
    norm = -np.log(2 * np.pi * iv(0, kappa))
    return lambda p, x: np.exp(norm[p] + kappa[p] * np.cos(np.asarray(x) - mu[p]))


def x0():
    return np.linspace(-np.pi, np.pi, NS0 + 1)[:-1]


def make(P, f, device_resident=False):
    from bayesian_quadrature_b200 import BatchBQ, PeriodicKernel
    x = x0()
    l0 = np.stack([f(p, x) for p in range(P)])
    return BatchBQ(np.tile(x, (P, 1)), l0, PARAMS_TL, PARAMS_L, seed=0, ns_reserve=ROUNDS, device_resident=device_resident,
                   kernel=PeriodicKernel, **OPT)


def rounds(P, f, device_resident):
    import torch
    bb = make(P, f, device_resident)
    grid = np.linspace(-np.pi, np.pi, NA)
    g_d = torch.from_numpy(grid).cuda()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(ROUNDS):
        if device_resident:
            idx, x_next = bb.choose_next(g_d, on_device=True)
            x_h = x_next.cpu().numpy()
            bb.add_observations(x_next, torch.from_numpy(np.array([f(p, x_h[p]) for p in range(P)])).cuda())
        else:
            idx, x_next = bb.choose_next(grid)
            bb.add_observations(x_next, np.array([f(p, x_next[p]) for p in range(P)]))
    torch.cuda.synchronize()
    s = time.perf_counter() - t0
    bb.sync_host()
    out = {"rounds_s": round(s, 4), "ms_per_round": round(1e3 * s / ROUNDS, 3), "ns_median_end": float(np.median(bb.ns)),
           "Z_mean_median": float(np.median(bb.Z_mean()))}
    bb.close()
    return out


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(1e3 * (time.perf_counter() - t0))
    return ts


def fit(P, f):
    bb = make(P, f)
    rows = bb._rows()
    htl, hl = rows[:, [0, 1, 6]], rows[:, [3, 4, 7]]
    ll0 = bb.log_lh(htl, hl, PARAMS)
    grad_ms = timed(lambda: bb.log_lh_grad(htl, hl, PARAMS), 10)
    llh_ms = timed(lambda: bb.log_lh(htl, hl, PARAMS), 10)
    t0 = time.perf_counter()
    res = bb.fit_hypers(PARAMS)
    fit_s = time.perf_counter() - t0
    out = {"log_lh_grad_ms": spread(grad_ms), "log_lh_ms": spread(llh_ms), "fit_s": round(fit_s, 3),
           "iterations_median": float(np.median(res["iterations"])), "iterations_max": int(res["iterations"].max()),
           "evaluations": int(res["evaluations"]), "converged": int(res["converged"].sum()),
           "log_lh_gain_median": round(float(np.median(res["log_lh"] - ll0)), 4),
           "period_tl_median": round(float(np.median(bb.period[:, 0])), 4)}
    bb.close()
    return out


def bq_loop(f, n):
    """The 20 fixed-hyper-parameter rounds of problems 0 .. n - 1 with one BQ object each: seconds."""
    from bayesian_quadrature_b200 import BQ, PeriodicKernel
    grid = np.linspace(-np.pi, np.pi, NA)
    t0 = time.perf_counter()
    for p in range(n):
        np.random.seed(p)
        x = x0()
        bq = BQ(x, f(p, x), kernel=PeriodicKernel, optim_method="L-BFGS-B", **OPT)
        bq.init(params_tl=PARAMS_TL, params_l=PARAMS_L)
        for _ in range(ROUNDS):
            x_a = float(grid[int(np.argmax(bq.expected_squared_mean(grid)))])
            bq.add_observation(x_a, float(f(p, x_a)))
        bq.Z_mean()
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--P", type=int, default=1024)
    ap.add_argument("--loop", type=int, default=8, help="problems of the BQ loop")
    a = ap.parse_args()
    from bayesian_quadrature_b200 import _lib
    _lib.load()
    if _lib.device_count() < 1:
        raise SystemExit("bench_batch_periodic.py: no CUDA device")
    P, f = a.P, likelihoods(a.P)
    name, power = card()
    head = {"bench": "batch_periodic", "gpu": name, "power_limit": power, "P": P, "ns0": NS0, "n_grid": 1000, "na": NA}
    rounds(min(P, 64), f, False)                      # warm-up: module loads and every launch shape of a round
    for mode in ("host", "device_resident"):
        r = rounds(P, f, mode == "device_resident")
        print("%s: %s" % (mode, r), file=sys.stderr, flush=True)
        print(json.dumps(dict(head, case="rounds_" + mode, rounds=ROUNDS, **r)), flush=True)
    r = fit(P, f)
    print("fit: %s" % r, file=sys.stderr, flush=True)
    print(json.dumps(dict(head, case="fit_hypers", params=PARAMS, **r)), flush=True)
    s = bq_loop(f, a.loop)
    print(json.dumps(dict(head, case="bq_loop", rounds=ROUNDS, problems=a.loop, seconds=round(s, 3),
                          extrapolated_to_P_s=round(s * P / a.loop, 1))), flush=True)


if __name__ == "__main__":
    main()
