#!/usr/bin/env python
"""BatchBQ.fit_hypers(["h", "w"]): the maximum-likelihood fit of every problem's hyper-parameters, with the value and
gradient of the joint log likelihood from one launch of the gradient kernel per optimiser step.  One JSON line per case on
stdout:

    python bench_fit_hypers.py > profiles/fit_hypers_r05.jsonl

Cases: P = 1024 problems at ns = 64 and P = 16384 at ns = 128 (BASELINE config C5), started at C5's hyper-parameters with
a fixed noise s = 0.1 (gp_log_l) and 1e-3 (gp_l): without noise the joint likelihood of these smooth problems keeps
growing as the Gram matrices become singular, and a fit ends wherever rounding stops it (DESIGN 8.2).  Reported per case:
  * one batched value-and-gradient evaluation of all P problems (BatchBQ.log_lh_grad) next to one BatchBQ.log_lh call
    (two setups of the batch: the proposal and the restore); both end in a device synchronise (results come back to the
    host), each shape is run once before it is timed;
  * the whole fit from the same start in every repetition: wall time, iterations per problem (median, max), problem
    evaluations, how many problems converged and the median gain of log_lh;
  * for context, the reference's path: BQ.fit_hypers (scipy, finite-difference gradients) looped over the first --loop
    problems, extrapolated linearly to P."""
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

PARAMS = ["h", "w"]
NOISE = (0.1, 1e-3)


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


def make(P, ns):
    from bayesian_quadrature_b200 import BatchBQ, synthetic
    x0, _ = synthetic.observations(ns)
    l0 = np.stack([synthetic.likelihood(ns, synthetic.problem_shift(p))(x0) for p in range(P)])
    opt = synthetic.options(ns)
    ptl, pl = synthetic.PARAMS_TL[:2] + (NOISE[0],), synthetic.PARAMS_L[:2] + (NOISE[1],)
    return BatchBQ(np.tile(x0, (P, 1)), l0, ptl, pl, opt["n_candidate"], opt["candidate_thresh"], opt["x_mean"], opt["x_var"],
                   seed=0), opt


def timed(f, reps):
    f()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        f()
        ts.append(1e3 * (time.perf_counter() - t0))
    return ts


def bq_loop(bb, opt, n):
    """BQ.fit_hypers of problems 0 .. n - 1 (same observations, candidates and start): (seconds, failures).  A call that
    raises "couldn't find good parameters" (its scipy restarts found no finite optimum) is timed as well."""
    from bayesian_quadrature_b200 import BQ, GaussianKernel
    t, failed = 0.0, 0
    for p in range(n):
        k, c = int(bb.ns[p]), int(bb.nc[p])
        bq = BQ(bb.x_s[p, :k].copy(), bb.l_s[p, :k].copy(), kernel=GaussianKernel, **opt)
        bq.init(params_tl=tuple(bb.hyp[p, :3]), params_l=tuple(bb.hyp[p, 3:]))
        bq.x_c, bq.nc = bb.x_c[p, :c].copy(), c
        t0 = time.perf_counter()
        try:
            bq.fit_hypers(PARAMS)
        except RuntimeError:
            failed += 1
        t += time.perf_counter() - t0
    return t, failed


def run(P, ns, reps, loop):
    bb, opt = make(P, ns)
    hyp0 = bb.hyp.copy()
    htl, hl = hyp0[:, :2], hyp0[:, 3:5]
    ll0 = bb.log_lh_grad(htl, hl, PARAMS)[0]
    grad_ms = timed(lambda: bb.log_lh_grad(htl, hl, PARAMS), 10)
    llh_ms = timed(lambda: bb.log_lh(htl, hl, PARAMS), 10)
    print("P=%d ns=%d: log_lh_grad %.2f ms, log_lh %.2f ms" % (P, ns, np.median(grad_ms), np.median(llh_ms)),
          file=sys.stderr, flush=True)
    fit_s, res = [], None
    for r in range(reps):
        bb.hyp[:] = hyp0
        t0 = time.perf_counter()
        res = bb.fit_hypers(PARAMS)
        fit_s.append(time.perf_counter() - t0)
        print("P=%d fit %d: %.2f s" % (P, r, fit_s[-1]), file=sys.stderr, flush=True)
    loop_s, loop_failed = bq_loop(bb, opt, loop)
    name, power = card()
    out = {
        "bench": "fit_hypers", "gpu": name, "power_limit": power, "P": P, "ns": ns, "params": PARAMS, "noise": NOISE,
        "capacity_class": int(bb._cap_class), "nc_median": float(np.median(bb.nc)),
        "log_lh_grad_ms": spread(grad_ms), "log_lh_ms": spread(llh_ms),
        "fit_s": spread(fit_s),
        "iterations_median": float(np.median(res["iterations"])), "iterations_max": int(res["iterations"].max()),
        "evaluations": int(res["evaluations"]), "converged": int(res["converged"].sum()),
        "log_lh_gain_median": round(float(np.median(res["log_lh"] - ll0)), 4),
        "bq_loop_problems": loop, "bq_loop_failed": loop_failed, "bq_loop_s": round(loop_s, 3), "bq_loop_extrapolated_s": round(loop_s * P / loop, 1),
    }
    bb.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--cases", default="1024x64,16384x128", help="comma-separated PxNS")
    ap.add_argument("--loop", type=int, default=8, help="problems of the BQ.fit_hypers loop")
    a = ap.parse_args()
    from bayesian_quadrature_b200 import _lib
    _lib.load()
    if _lib.device_count() < 1:
        raise SystemExit("bench_fit_hypers.py: no CUDA device")
    for case in a.cases.split(","):
        P, ns = (int(v) for v in case.split("x"))
        print(json.dumps(run(P, ns, a.reps, a.loop)), flush=True)


if __name__ == "__main__":
    main()
