#!/usr/bin/env python
"""BatchBQ.marginalize and choose_next(deterministic=False): the quantities of every problem under S hyper-parameter sets
per problem, and the reference's random tie-break on the device.  One JSON line per case on stdout:

    python bench_batch_marginalize.py > profiles/batch_marginalize_r09.jsonl

Cases: P = 1024 problems at ns = 64 and P = 16384 at ns = 128 (BASELINE config C5), S = 16 sets per problem from the C4
ranges (synthetic.hyper_sets, as bench_batch_marginal.py times the loss: no sampler failure enters the timing), a sorted
4096-point grid.  Timed: marginalize(["Z_mean", "Z_var"]) (the setup phase alone), marginalize([("expected_Z_var", x)],
on_device=True) next to marginal_loss on the same sets, marginalize([("l_mean", x)]), one choose_next(deterministic=False)
round next to a deterministic one (same sets), and the tie kernel alone over a [P, na] loss (larger than L2 at C5; one more read of
it after the argmin).  For context, a loop of BQ.marginalize over 8 problems, extrapolated linearly to P.  Every timing is
the median (with min / max) of repeated calls, each ending in a device synchronise, after one untimed call."""
import argparse
import json
import os
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
warnings.simplefilter("ignore")

from bench_batch_marginal import PARAMS, card, make, spread      # noqa: E402


def timed(fn, reps):
    import torch
    fn()
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(1e3 * (time.perf_counter() - t0))
    return spread(ts)


def bq_loop(bb, grid, htl, hl, n_problems=8):
    """Seconds of BQ.marginalize([Z_mean, Z_var, expected_Z_var]) over the first problems, their samples given."""
    from bayesian_quadrature_b200 import BQ, GaussianKernel, synthetic
    ns = int(bb.ns[0])
    opt = synthetic.options(ns)
    t = 0.0
    for p in range(n_problems):
        bq = BQ(bb.x_s[p, :ns].copy(), bb.l_s[p, :ns].copy(), kernel=GaussianKernel, **opt)
        bq.init(params_tl=synthetic.PARAMS_TL, params_l=synthetic.PARAMS_L)
        bq.sample_hypers = lambda params, n=1, nburn=10, p=p: (htl[p], hl[p])
        t0 = time.perf_counter()
        bq.marginalize([bq.Z_mean, bq.Z_var, lambda: bq.expected_Z_var(grid)], htl.shape[1], PARAMS)
        t += time.perf_counter() - t0
    return t


def run(P, ns, S, reps):
    import torch
    from bayesian_quadrature_b200 import synthetic
    bb, grid = make(P, ns)
    x_d = torch.from_numpy(grid).cuda()
    h = synthetic.hyper_sets(P * S).reshape(P, S, 4)
    hyp = (np.ascontiguousarray(h[..., :2]), np.ascontiguousarray(h[..., 2:]))
    kw = dict(params=PARAMS, hypers=hyp)
    out = {"bench": "batch_marginalize", "P": P, "ns": ns, "S": S, "na": int(grid.size), "capacity_class": int(bb._cap_class),
           "reps": reps}
    out["scalars_ms"] = timed(lambda: bb.marginalize(["Z_mean", "Z_var"], **kw), reps)
    out["expected_Z_var_on_device_ms"] = timed(lambda: bb.marginalize([("expected_Z_var", x_d)], on_device=True, **kw), reps)
    out["marginal_loss_ms"] = timed(lambda: bb.marginal_loss(x_d, hyp[0], hyp[1], PARAMS), reps)
    out["l_mean_on_device_ms"] = timed(lambda: bb.marginalize([("l_mean", x_d)], on_device=True, **kw), reps)
    out["choose_next_deterministic_ms"] = timed(lambda: bb.choose_next(x_d, on_device=True, **kw), reps)
    out["choose_next_random_ms"] = timed(lambda: bb.choose_next(x_d, on_device=True, deterministic=False, seed=1, **kw), reps)
    # the tie kernel alone over a [P, na] loss matrix larger than L2: a smooth row with ties near its minimum
    loss = -torch.cos(torch.linspace(0, 3, grid.size, dtype=torch.float64, device="cuda"))[None, :].repeat(P, 1)
    loss += 1e-9 * torch.rand(P, 1, dtype=torch.float64, device="cuda")
    mins = torch.empty(P, dtype=torch.float64, device="cuda")
    idxs = torch.empty(P, dtype=torch.int64, device="cuda")
    cnts = torch.empty(P, dtype=torch.int64, device="cuda")
    u = torch.rand(P, dtype=torch.float64, device="cuda")
    bb.batch.argmin_rows_device(loss, mins, idxs)
    out["argmin_rows_ms"] = timed(lambda: bb.batch.argmin_rows_device(loss, mins, idxs), reps * 4)
    out["tie_kernel_ms"] = timed(lambda: bb.batch.argmin_ties_rows_device(loss, mins, u, idxs, cnts), reps * 4)
    out["tie_kernel_loss_MB"] = round(8 * P * grid.size / 2 ** 20, 1)
    out["tie_kernel_GBps_one_read"] = round(8 * P * grid.size / (out["tie_kernel_ms"]["median"] * 1e-3) / 1e9, 1)
    out["ties_per_row"] = spread(cnts.cpu().numpy())
    t8 = bq_loop(bb, grid, hyp[0], hyp[1])
    out["bq_marginalize_loop_8_problems_s"] = round(t8, 3)
    out["bq_marginalize_loop_extrapolated_to_P_s"] = round(t8 * P / 8, 1)
    out["gpu"], out["power_limit"] = card()
    bb.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cases", default="1024x64,16384x128", help="comma-separated PxNS")
    ap.add_argument("--samples", type=int, default=16)
    a = ap.parse_args()
    from bayesian_quadrature_b200 import _lib
    _lib.load()
    if _lib.device_count() < 1:
        raise SystemExit("bench_batch_marginalize.py: no CUDA device")
    for case in a.cases.split(","):
        P, ns = (int(v) for v in case.split("x"))
        print(json.dumps(run(P, ns, a.samples, a.reps)), flush=True)


if __name__ == "__main__":
    main()
