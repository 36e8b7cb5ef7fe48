#!/usr/bin/env python
"""BatchBQ's per-point read-outs at P = 1024 problems of ns = 64 and at C5 (P = 16384, ns = 128), on a shared 4096-point
grid.  One JSON line per case on stdout:

    python bench_batch_readout.py > profiles/batch_readout_r07.jsonl

Reported, each the median (min-max) of --reps timed calls after one untimed call, every call ending in a device
synchronise:
  * expected_Z_var(on_device=True) of all problems next to the bare scoring pass of choose_next (score_device of all P
    problems into a [P, na] buffer), and the row-wise expected-variance kernel alone over that buffer (HBM-resident, in
    the chunks expected_Z_var uses; inside expected_Z_var each chunk is still in L2);
  * l_mean and l_var (on_device=True): the prediction kernel for all problems;
  * for context, a loop of BQ.expected_Z_var over the first --loop problems with one BQ object each, extrapolated to P."""
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
CASES = [(1024, 64), (16384, 128)]


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


def make(P, ns):
    from bayesian_quadrature_b200 import BatchBQ, synthetic
    x0, _ = synthetic.observations(ns)
    l0 = np.stack([synthetic.likelihood(ns, synthetic.problem_shift(p))(x0) for p in range(P)])
    opt = synthetic.options(ns)
    return BatchBQ(np.tile(x0, (P, 1)), l0, synthetic.PARAMS_TL, synthetic.PARAMS_L, opt["n_candidate"], opt["candidate_thresh"],
                   opt["x_mean"], opt["x_var"], seed=0)


def case(P, ns, reps):
    import torch
    from bayesian_quadrature_b200 import synthetic
    bb = make(P, ns)
    grid = synthetic.query_grid(ns, NA)
    g = torch.from_numpy(grid).cuda()
    esm = torch.empty(P, NA, dtype=torch.float64, device="cuda")
    out = torch.empty_like(esm)
    flags = torch.zeros(P, dtype=torch.int32, device="cuda")
    per = max(1, min(P, bb.LOSS_CHUNK_BYTES // (8 * NA)))

    def rows_kernel():
        for q0 in range(0, P, per):
            cq = min(per, P - q0)
            bb.batch.expected_var_rows_device(q0, cq, esm[q0:q0 + cq], out[q0:q0 + cq])
    score = timed(lambda: bb.batch.score_device(g, esm, None, None, flags), reps)
    ev_kernel = timed(rows_kernel, reps)
    ev = timed(lambda: bb.expected_Z_var(g, on_device=True), reps)
    ev_d = bb.expected_Z_var(g, on_device=True)
    assert torch.equal(ev_d, out), "expected_Z_var differs from the kernel over the full score buffer"
    l_mean = timed(lambda: bb.l_mean(g, on_device=True), reps)
    l_var = timed(lambda: bb.l_var(g, on_device=True), reps)
    res = {"score_device_ms": spread(score), "expected_Z_var_ms": spread(ev), "expected_var_rows_kernel_ms": spread(ev_kernel),
           "expected_Z_var_over_score": round(float(np.median(ev) / np.median(score)), 4),
           "rows_kernel_over_score": round(float(np.median(ev_kernel) / np.median(score)), 4),
           "l_mean_ms": spread(l_mean), "l_var_ms": spread(l_var), "chunk_problems": per,
           "expected_Z_var_evals_per_s": round(P * NA / (np.median(ev) / 1e3), 1)}
    bb.close()
    return res


def bq_loop(ns, n):
    """BQ.expected_Z_var on the same grid for problems 0 .. n - 1, one BQ object each (init not timed): seconds."""
    from bayesian_quadrature_b200 import BQ, GaussianKernel, synthetic
    grid = synthetic.query_grid(ns, NA)
    bqs = [synthetic.make_bq(BQ, GaussianKernel, ns, shift=synthetic.problem_shift(p), seed=p) for p in range(n)]
    bqs[0].expected_Z_var(grid)
    t0 = time.perf_counter()
    for bq in bqs:
        bq.expected_Z_var(grid)
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--loop", type=int, default=8, help="problems of the BQ loop")
    ap.add_argument("--small", action="store_true", help="P = 64 and 256 instead of 1024 and 16384 (a quick check)")
    a = ap.parse_args()
    from bayesian_quadrature_b200 import _lib
    _lib.load()
    if _lib.device_count() < 1:
        raise SystemExit("bench_batch_readout.py: no CUDA device")
    name, power = card()
    for P, ns in ([(64, 64), (256, 128)] if a.small else CASES):
        head = {"bench": "batch_readout", "gpu": name, "power_limit": power, "P": P, "ns": ns, "na": NA}
        r = case(P, ns, a.reps)
        print("P=%d ns=%d: %s" % (P, ns, r), file=sys.stderr, flush=True)
        print(json.dumps(dict(head, case="readout", **r)), flush=True)
        s = bq_loop(ns, a.loop)
        print(json.dumps(dict(head, case="bq_loop", problems=a.loop, seconds=round(s, 5),
                              extrapolated_to_P_s=round(s * P / a.loop, 3))), flush=True)


if __name__ == "__main__":
    main()
