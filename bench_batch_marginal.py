#!/usr/bin/env python
"""One marginalised active-sampling round of BatchBQ (choose_next(x_a, n=S, params=["h", "w"])): the batched slice
sampler (one log-density launch of all P problems per step), then the marginal loss of the P x S (problem, sample)
instances -- chunked setup, grouped scoring, segmented sample reduction -- and the per-problem argmin.  One JSON line per
case on stdout:

    python bench_batch_marginal.py > profiles/batch_marginal_r04.jsonl

Cases: P = 1024 problems at ns = 64 and P = 16384 at ns = 128 (BASELINE config C5), S = 16 samples, a 4096-point grid.
Every timing ends in a device synchronise (the log density copies its results to the host) or is taken with CUDA events;
each shape is run once before it is timed, and repeated measurements are reported as min / median / max.  The chains of a
round advance in lock-step, so its slowest chain sets its length: a round is capped at --steps-per-sample x (S + 1)
log-density steps, and the line reports how many chains the cap stopped (util.slice_sample_batch, max_steps)."""
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
L2_BYTES = 126 << 20
COPY_TBS = 6.55          # device-to-device copy rate measured on the B200 (DESIGN.md 4.5)


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
    return BatchBQ(np.tile(x0, (P, 1)), l0, synthetic.PARAMS_TL, synthetic.PARAMS_L, opt["n_candidate"], opt["candidate_thresh"],
                   opt["x_mean"], opt["x_var"], seed=0), synthetic.query_grid(ns, 4096)


def events():
    import torch
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def reduction_hbm(bb, S, na, gbytes=2.0):
    """The segmented reduction over an esm buffer far larger than L2 (HBM-bound rate)."""
    import torch
    G = int(gbytes * 1e9 // (8 * S * na))
    esm = torch.rand(G * S, na, dtype=torch.float64, device="cuda") - 0.5
    acc = torch.zeros(G, na, dtype=torch.float64, device="cuda")
    bb.batch.sum_neg_accum_groups_device(esm, G, S, acc)
    ts = []
    for _ in range(10):
        a, b = events()
        a.record()
        bb.batch.sum_neg_accum_groups_device(esm, G, S, acc)
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b) / 1e3)
    nbytes = 8 * G * na * (S + 2)
    del esm, acc
    return nbytes, [nbytes / t / 1e9 for t in ts]


def run(P, ns, S, reps, steps_per_sample):
    import torch
    from bayesian_quadrature_b200 import synthetic
    bb, grid = make(P, ns)
    x_d = torch.from_numpy(grid).cuda()
    max_steps = steps_per_sample * (S + 1)
    step_s = []
    log_lh = bb.log_lh

    def timed_log_lh(*a):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = log_lh(*a)                                      # ends by copying its results to the host
        step_s.append(time.perf_counter() - t0)
        if len(step_s) % 250 == 0:
            print("P=%d step %d: %.2f ms" % (P, len(step_s), 1e3 * step_s[-1]), file=sys.stderr, flush=True)
        return r

    bb.log_lh = timed_log_lh
    # sampled sets can reach Gram matrices so ill-conditioned that some expected squared mean is invalid; marginal_loss
    # then raises, as BQ.marginal_loss does.  The loss of such a round is timed on S sets per problem from the
    # well-conditioned C4 ranges (synthetic.hyper_sets; same shapes, same work) and the JSON line says so.
    c4 = synthetic.hyper_sets(P * S).reshape(P, S, 4)
    c4 = (np.ascontiguousarray(c4[..., :2]), np.ascontiguousarray(c4[..., 2:]))
    bb.sample_hypers(PARAMS, n=1, nburn=1, max_steps=steps_per_sample)   # warm-up of every shape
    bb.choose_next(x_d, hypers=c4, params=PARAMS)
    print("P=%d ns=%d: warm-up done" % (P, ns), file=sys.stderr, flush=True)
    rounds, sampler_s, n_steps, unfinished, sampled_ok, errors, step_ms = [], [], [], [], [], [], []
    for r in range(reps):
        step_s.clear()
        st = {}
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        hyp = bb.sample_hypers(PARAMS, n=S, nburn=1, seed=r, max_steps=max_steps, stats=st)
        t1 = time.perf_counter()
        sampler_s.append(t1 - t0)
        try:
            idx, _ = bb.choose_next(x_d, hypers=hyp, params=PARAMS)
            sampled_ok.append(True)
        except RuntimeError as e:
            sampled_ok.append(False)
            errors.append(str(e))
            hyp = c4
            t1 = time.perf_counter()                         # the failed attempt is not part of the round
            idx, _ = bb.choose_next(x_d, hypers=hyp, params=PARAMS)
        t2 = time.perf_counter()                             # choose_next returns host arrays: synchronised
        rounds.append(sampler_s[-1] + (t2 - t1))
        n_steps.append(st["steps"])
        unfinished.append(int(st["unfinished"].size))
        step_ms += [1e3 * v for v in step_s]
        print("P=%d round %d: %.2f s, %d steps, %d chains stopped by the cap" % (P, r, rounds[-1], st["steps"], unfinished[-1]),
              file=sys.stderr, flush=True)
    htl, hl = hyp
    loss_ms, ph = [], []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        bb.marginal_loss(x_d, htl, hl, PARAMS)
        torch.cuda.synchronize()
        loss_ms.append(1e3 * (time.perf_counter() - t0))
    for _ in range(reps):                                    # phases in runs of their own: the events synchronise
        t = {}
        bb.marginal_loss(x_d, htl, hl, PARAMS, timings=t)
        ph.append(t)
    per_setup, per_score = bb._chunks(S, grid.size)
    esm_bytes = 8 * per_score * S * grid.size
    red_bytes = 8 * P * grid.size * (S + 2)                  # esm read once, acc read and written once
    hbm_bytes, hbm_gbs = reduction_hbm(bb, S, grid.size)
    name, power = card()
    out = {
        "bench": "batch_marginal", "gpu": name, "power_limit": power, "P": P, "ns": ns, "S": S, "na": int(grid.size),
        "capacity_class": int(bb._cap_class), "reps": reps, "max_sampler_steps": max_steps,
        "round_s": spread(rounds),
        "sampler_s": spread(sampler_s),
        "sampler_steps": spread(n_steps),
        "sampler_steps_per_sample": spread(np.asarray(n_steps) / S),
        "chains_stopped_by_cap": unfinished,
        "log_lh_step_ms": spread(step_ms),
        "marginal_loss_ms": spread(loss_ms),
        "loss_setup_ms": spread([1e3 * t["setup"] for t in ph]),
        "loss_score_ms": spread([1e3 * t["score"] for t in ph]),
        "loss_reduce_ms": spread([1e3 * t["reduce"] for t in ph]),
        "problems_per_setup_chunk": per_setup, "problems_per_score_launch": per_score,
        "esm_chunk_MB": round(esm_bytes / 2 ** 20, 1), "esm_chunk_fits_l2": bool(esm_bytes <= L2_BYTES),
        "reduce_GBps_in_loop": spread([red_bytes / t["reduce"] / 1e9 for t in ph]),
        "reduce_GBps_hbm": spread(hbm_gbs), "reduce_hbm_bytes_GB": round(hbm_bytes / 1e9, 2),
        "reduce_hbm_share_of_copy": round(float(np.median(hbm_gbs)) / (COPY_TBS * 1e3), 3),
        "sampled_sets_scored": sampled_ok, "sampled_set_errors": errors[:2],
        "choice_checksum": int(np.asarray(idx).sum()),
    }
    bb.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cases", default="1024x64,16384x128", help="comma-separated PxNS")
    ap.add_argument("--samples", type=int, default=16)
    ap.add_argument("--steps-per-sample", type=int, default=100,
                    help="cap of a round's log-density steps, per iteration of the chains (the slowest chain sets a round)")
    a = ap.parse_args()
    from bayesian_quadrature_b200 import _lib
    _lib.load()
    if _lib.device_count() < 1:
        raise SystemExit("bench_batch_marginal.py: no CUDA device")
    for case in a.cases.split(","):
        P, ns = (int(v) for v in case.split("x"))
        print(json.dumps(run(P, ns, a.samples, a.reps, a.steps_per_sample)), flush=True)


if __name__ == "__main__":
    main()
