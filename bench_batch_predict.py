#!/usr/bin/env python
"""BatchBQ.l_mean + l_var (on_device=True) on a shared 4096-point grid for the problems the scoring kernels' prediction mode
does not serve -- the periodic kernel, a noisy gp_l, the 512 class -- which go through the prediction kernel
(csrc/bq_predict.cu).  One JSON line per case on stdout:

    python bench_batch_predict.py > profiles/batch_predict_r08.jsonl

Cases:
  * periodic: P = 1024 problems of bench_batch_periodic.py (von Mises likelihoods, ns0 = 16, s_l = 1e-3), grid [-pi, pi);
  * c5_noisy: P = 16384 C5 problems (ns = 128) with s_l = 1e-3, and next to it c5_mode2, the same batch with s_l = 0, which
    takes the scoring kernels' prediction mode;
  * class512: P = 64 problems of ns = 300 (the plain-FP64 path of the 512 class).
Reported, each the median (min-max) of --reps timed calls after one untimed call, every call ending in a device
synchronise: l_mean + l_var together (two prediction passes and the product), l_mean alone, and the bare prediction launch
over all P problems (predict_rows_device, or predict_device for c5_mode2) with the point evaluations per second it reaches.
For context, the host-GP route the batch took before (gp_l.mean and np.diag(gp_log_l.cov) on BatchBQ._host_gps) over the
first --loop problems, extrapolated linearly to P: labelled ``extrapolated_to_P_s``."""
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

NA = 4096


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


def timed(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(1e3 * (time.perf_counter() - t0))
    return ts


def periodic(P):
    from bayesian_quadrature_b200 import BatchBQ, PeriodicKernel
    from bench_batch_periodic import NS0, OPT, PARAMS_L, PARAMS_TL, likelihoods
    f = likelihoods(P)
    x = np.linspace(-np.pi, np.pi, NS0 + 1)[:-1]
    bb = BatchBQ(np.tile(x, (P, 1)), np.stack([f(p, x) for p in range(P)]), PARAMS_TL, PARAMS_L, seed=0,
                 kernel=PeriodicKernel, **OPT)
    return bb, np.linspace(-np.pi, np.pi, NA + 1)[:-1]


def gaussian(P, ns, s_l):
    from bayesian_quadrature_b200 import BatchBQ, synthetic
    x0, _ = synthetic.observations(ns)
    l0 = np.stack([synthetic.likelihood(ns, synthetic.problem_shift(p))(x0) for p in range(P)])
    opt = synthetic.options(ns)
    bb = BatchBQ(np.tile(x0, (P, 1)), l0, synthetic.PARAMS_TL, synthetic.PARAMS_L[:2] + (s_l,), opt["n_candidate"],
                 opt["candidate_thresh"], opt["x_mean"], opt["x_var"], seed=0)
    return bb, synthetic.query_grid(ns, NA)


def case(bb, grid, reps, mode2):
    import torch
    P = bb.P
    g = torch.from_numpy(grid).cuda()
    m = torch.empty(P, NA, dtype=torch.float64, device="cuda")
    v = torch.empty_like(m)
    launch = (lambda: bb.batch.predict_device(g, m, v)) if mode2 else (lambda: bb.batch.predict_rows_device(g, m, v))
    kernel = timed(launch, reps)
    both = timed(lambda: (bb.l_mean(g, on_device=True), bb.l_var(g, on_device=True)), reps)
    mean = timed(lambda: bb.l_mean(g, on_device=True), reps)
    return {"l_mean_plus_l_var_ms": spread(both), "l_mean_ms": spread(mean), "prediction_launch_ms": spread(kernel),
            "launch_points_per_s": round(P * NA / (np.median(kernel) / 1e3), 1)}


def host_route(bb, grid, n):
    """BatchBQ's former route for one problem (host GPs, np.diag of the [na, na] covariance) over problems 0 .. n - 1: s."""
    t0 = time.perf_counter()
    for p in range(n):
        gp_log_l, gp_l = bb._host_gps(p)
        gp_l.mean(grid)
        np.diag(gp_log_l.cov(grid)).copy()
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--loop", type=int, default=8, help="problems of the host-GP route")
    ap.add_argument("--small", action="store_true", help="P = 64 / 256 / 8 instead of 1024 / 16384 / 64 (a quick check)")
    a = ap.parse_args()
    from bayesian_quadrature_b200 import _lib
    _lib.load()
    if _lib.device_count() < 1:
        raise SystemExit("bench_batch_predict.py: no CUDA device")
    name, power = card()
    p_per, p_c5, p_512 = (64, 256, 8) if a.small else (1024, 16384, 64)
    cases = [("periodic", lambda: periodic(p_per), False, 16),
             ("c5_noisy", lambda: gaussian(p_c5, 128, 1e-3), False, 128),
             ("c5_mode2", lambda: gaussian(p_c5, 128, 0.0), True, 128),
             ("class512", lambda: gaussian(p_512, 300, 0.0), False, 300)]
    for label, make, mode2, ns in cases:
        bb, grid = make()
        head = {"bench": "batch_predict", "gpu": name, "power_limit": power, "case": label, "P": bb.P, "ns": ns, "na": NA,
                "s_l": float(bb.hyp[0, 5]), "capacity_class": int(bb._cap_class),
                "route": "prediction mode of the scoring kernels" if mode2 else "prediction kernel"}
        r = case(bb, grid, a.reps, mode2)
        print("%s: %s" % (label, r), file=sys.stderr, flush=True)
        print(json.dumps(dict(head, **r)), flush=True)
        if not mode2:
            s = host_route(bb, grid, a.loop)
            print(json.dumps(dict(head, case=label + "_host_gps", route="host GPs (extrapolated)", problems=a.loop,
                                  seconds=round(s, 4), extrapolated_to_P_s=round(s * bb.P / a.loop, 2))), flush=True)
        bb.close()


if __name__ == "__main__":
    main()
