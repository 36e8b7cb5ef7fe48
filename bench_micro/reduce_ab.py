#!/usr/bin/env python
"""A/B timing of the reduction entry points (csrc/bq_reduce.cu) of two or more builds of libbq_b200.so.

    python bench_micro/reduce_ab.py --lib A.so --lib B.so [--lib C.so ...] [--runs 3] [--reps 20] [--out FILE]

Every run is a fresh process with BQB200_LIB set to one library, and the libraries alternate run by run (A B A B ...), so
that drift of the shared machine falls on all of them.  Each entry point is timed with CUDA events around one call after
warm-up (expected_var_host, which ends in a host synchronise, with the host clock), and the 126 MB L2 is overwritten by a
256 MB write before every repetition.  A run reports the median over its repetitions; the summary gives, per library, the median
and the spread (max - min) over runs in microseconds, with the card's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def worker(reps, warmup):
    sys.path.insert(0, ROOT)
    import torch
    from bayesian_quadrature_b200 import BQ, GaussianKernel, _lib, synthetic

    dev = torch.device("cuda")
    g = torch.Generator(device="cuda").manual_seed(7)

    def rand(*shape):
        return torch.rand(*shape, dtype=torch.float64, device=dev, generator=g) - 0.5

    flush = torch.empty(32 * 2 ** 20, dtype=torch.float64, device=dev)        # 256 MB > 126 MB of L2

    def timed(fn, host_clock=False):
        for _ in range(warmup):
            fn()
        ts = []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for r in range(reps):
            flush.fill_(r)
            torch.cuda.synchronize()
            if host_clock:
                t0 = time.perf_counter()
                fn()
                ts.append((time.perf_counter() - t0) * 1e6)
            else:
                e0.record()
                fn()
                e1.record()
                e1.synchronize()
                ts.append(e0.elapsed_time(e1) * 1e3)
        return float(np.median(ts))

    # one set-up instance (ns = 64) for the entry points that read Z_mean / Z_var
    ns = 64
    bq = synthetic.make_bq(BQ, GaussianKernel, ns)
    opt = synthetic.options(ns)
    b1 = _lib.Batch(1, ns)
    info = b1.setup([ns], [bq.nc], bq.x_s[None], bq.l_s[None], bq.x_c[None], [synthetic.PARAMS_TL + synthetic.PARAMS_L],
                    [[opt["x_mean"], opt["x_var"], opt["candidate_thresh"]]])
    assert info["status"][0] == 0
    res = {}

    b = _lib.Batch(1024, 16)                          # mean_neg_device reduces n_inst rows
    esm, loss = rand(1024, 10 ** 5), torch.empty(10 ** 5, dtype=torch.float64, device=dev)
    res["mean_neg_device 1024x1e5"] = timed(lambda: b.mean_neg_device(esm, loss))
    b.close()
    del esm

    esm, acc = rand(74, 10 ** 5), torch.zeros(10 ** 5, dtype=torch.float64, device=dev)   # bench.py C4: 74-instance chunks
    res["sum_neg_accum_device 74x1e5"] = timed(lambda: b1.sum_neg_accum_device(esm, 74, acc))
    esm, acc = rand(8 * 64, 10 ** 4), torch.zeros(8, 10 ** 4, dtype=torch.float64, device=dev)
    res["sum_neg_accum_groups_device 8x64x1e4"] = timed(lambda: b1.sum_neg_accum_groups_device(esm, 8, 64, acc))

    esm, out = rand(10 ** 7), torch.empty(10 ** 7, dtype=torch.float64, device=dev)
    res["expected_var_device 1e7"] = timed(lambda: b1.expected_var_device(0, esm, out))
    del esm, out
    x = synthetic.query_grid(ns, 10 ** 6)
    res["expected_var_host pageable 1e6"] = timed(lambda: b1.expected_var_host(x), host_clock=True)

    pair = torch.empty(2, dtype=torch.float64, device=dev)
    for n in (10 ** 6, 10 ** 7):
        v = rand(n)
        res["argmin_device %.0e" % n] = timed(lambda: b1.argmin_device(v))
        res["argmin_pair_device %.0e" % n] = timed(lambda: b1.argmin_pair_device(v, 0, pair))
    del v

    b = _lib.Batch(16384, 16)                         # argmin_rows_device reduces n_inst rows
    v = rand(16384, 4096)
    mins = torch.empty(16384, dtype=torch.float64, device=dev)
    idxs = torch.empty(16384, dtype=torch.int64, device=dev)
    res["argmin_rows_device 16384x4096"] = timed(lambda: b.argmin_rows_device(v, mins, idxs))
    b.close()
    b1.close()
    print(json.dumps(res))


def gpu_name_and_power():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              stdout=subprocess.PIPE, text=True, check=True).stdout.strip()
    except (OSError, subprocess.CalledProcessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], help="a libbq_b200.so; give two or more")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", help="also write the summary here (JSON)")
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        worker(args.reps, args.warmup)
        return
    if len(args.lib) < 2:
        raise SystemExit("give two or more libraries: --lib A.so --lib B.so ...")
    runs = {lib: [] for lib in args.lib}
    for _ in range(args.runs):
        for lib in args.lib:
            env = dict(os.environ, BQB200_LIB=os.path.abspath(lib))
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", "--reps", str(args.reps),
                                "--warmup", str(args.warmup)], env=env, stdout=subprocess.PIPE, text=True, check=True)
            runs[lib].append(json.loads(r.stdout.strip().splitlines()[-1]))
    summary = {"gpu": gpu_name_and_power(), "runs": args.runs, "reps": args.reps, "unit": "us", "libs": args.lib, "cases": {}}
    print("%s; %d runs each, median of %d repetitions per run (us); ratio = median / median of the first library" % (
        summary["gpu"], args.runs, args.reps))
    for i, lib in enumerate(args.lib):
        print("  [%d] %s" % (i, lib))
    print("%-40s" % "entry point" + "".join("%22s" % ("[%d] median spread ratio" % i) for i in range(len(args.lib))))
    for case in runs[args.lib[0]][0]:
        rows = []
        for lib in args.lib:
            v = [r[case] for r in runs[lib]]
            rows.append({"median": float(np.median(v)), "spread": max(v) - min(v), "runs": v})
        summary["cases"][case] = rows
        print("%-40s" % case + "".join("%10.2f %5.2f %5.3f" % (r["median"], r["spread"], r["median"] / rows[0]["median"])
                                       for r in rows))
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(summary, fh, indent=1)


if __name__ == "__main__":
    main()
