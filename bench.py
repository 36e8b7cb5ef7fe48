#!/usr/bin/env python
"""bench.py — expected_Z_var query-point evaluations per second on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle/_ref)
    python bench.py ... --dump-outputs DIR                   # + the last timed step's outputs as DIR/*.npy

Workload (config.workload): BASELINE.json configs[1] — 1-D BQ, 64 observations, expected_Z_var over
a 10^6-point grid (SURVEY.md §8(d) generator).  A *step* is one pass of the hot path over the
grid: the scoring kernel (esm for every point, expected variance Zm^2 + Zv - esm in its epilogue,
per-CTA minima) and one small kernel that reduces them to the deterministic (min, first index)
choose_next needs and — at N > 1 — exchanges the ranks' pairs over peer-mapped memory (NCCL
all-gather if symmetric memory is unavailable); the result lands in page-locked host memory.  At
N > 1 every rank scores 10^6 points of an N x 10^6 grid (weak scaling, block-cyclic shards).  The
per-hyper-set setup kernel (Gram, Cholesky, Z_mean, Z_var — amortised over the grid, SURVEY §8(d))
is timed separately (setup_ms).

Timing: W warm-up steps, then K steps enqueued back to back between a barrier + synchronize on both
sides, each bracketed by CUDA events on the launching stream; cold L2 through eight rotating 24 MB
input/output sets (192 MB > 126 MB of L2); max over ranks.  `value` is device-resident throughput
(inputs already in HBM); `e2e` is the same pass through the public host API (BQ.expected_Z_var) with
page-locked host buffers, the host-to-device and device-to-host traffic inside the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NS = 64
NA = 10 ** 6
METRIC = "expected_Z_var candidate evals/sec"
UNIT = "evals/s"


def w_flop(ns, nc):
    """Algorithmic FP64 flops per evaluation (SURVEY.md §8(d))."""
    n = ns + nc
    return n * n + ns * ns + 2 * (3 * n + 2 * ns) + 40


def w_exp(ns, nc):
    return ns + nc + ns + 4


def fp64_peak_tflops():
    """FP64 roofline denominator.  MEASURED_PEAKS.json carries no FP64 figure, so the peak is this
    repo's own microbenchmark (bench_micro/fp64_peaks.cu, DMMA m8n8k4 on all SMs), committed as
    profiles/fp64_peaks_r01.json."""
    p = os.path.join(ROOT, "profiles", "fp64_peaks_r01.json")
    try:
        with open(p) as fh:
            d = json.load(fh)
        return max(v for k, v in d.items() if k.startswith("dmma") or k.startswith("dfma")), "measured:profiles/fp64_peaks_r01.json"
    except Exception:
        return 37.2, "nominal:148 SM x 64 DFMA/clk x 1.965 GHz"


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the scoring kernel on the bench workload, from the
    committed `ncu --set full` capture (profiles/ncu_score_traffic.json, written by profiles/summarize.py)."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_score_traffic.json")) as fh:
            d = json.load(fh)
        return float(d["dram_bytes_read"]) + float(d["dram_bytes_write"])
    except Exception:
        return None


class ClockSampler(object):
    """`nvidia-smi -lms 200` in its own process for the duration of the timed regions (the profiling
    recipe's clocks line); parsed when stopped.  A separate process, so it never holds this process's GIL."""

    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.path = "/tmp/bq_b200_clocks_%d_%d.csv" % (os.getpid(), index)
        self.fh = open(self.path, "w")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.fh, stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def start(self):
        return self

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        self.fh.close()
        rows = [[c.strip() for c in line.split(",")] for line in open(self.path) if line.strip()]
        os.unlink(self.path)

        def num(v):
            try:
                return float(v)
            except ValueError:
                return None
        sm = [num(r[0]) for r in rows if num(r[0]) is not None]
        mx = [num(r[1]) for r in rows if len(r) > 1 and num(r[1]) is not None]
        pw = [num(r[2]) for r in rows if len(r) > 2 and num(r[2]) is not None]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in rows for i in range(4) if len(r) > 3 + i and r[3 + i].lower() == "active"})
        # "under load": samples at or above half the maximum clock (idle samples between phases are dropped)
        load = [v for v in sm if mx and v >= 0.5 * max(mx)] or sm
        return {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": reasons, "samples": len(rows)}


def build_problem():
    """C2 inputs.  The candidate draw uses the host RNG exactly like BQ.init (bq.py:967-991)."""
    from bayesian_quadrature_b200 import synthetic
    from bayesian_quadrature_b200.bq import BQ
    from bayesian_quadrature_b200.gp import GaussianKernel
    bq = synthetic.make_bq(BQ, GaussianKernel, NS)
    return bq


# ------------------------------------------------------------------------------------------ reference arm
def _ref_worker(args):
    lo, hi, na_total = args
    os.environ["OPENBLAS_NUM_THREADS"] = "1"
    import warnings
    warnings.simplefilter("ignore")
    from oracle import build_ref
    from bayesian_quadrature_b200 import synthetic
    bqmod, gp = build_ref.import_reference()
    bq = synthetic.make_bq(bqmod.BQ, gp.GaussianKernel, NS)
    x_a = synthetic.query_grid(NS, na_total)[lo:hi]
    t0 = time.perf_counter()
    ev = bq.expected_Z_var(x_a)
    return time.perf_counter() - t0, float(ev.sum())


def reference_pass(cores, pts_per_core):
    """One bounded sample of the C2 workload on the reference's own CPU implementation: `cores`
    forked processes each score a contiguous slice of the 10^6 grid (the reference itself is single
    threaded; this is the most favourable multi-core use of it, BASELINE.md §3)."""
    import multiprocessing as mp
    starts = np.linspace(0, NA - pts_per_core, cores).astype(np.int64)
    jobs = [(int(s), int(s) + pts_per_core, NA) for s in starts]
    ctx = mp.get_context("fork")
    t0 = time.perf_counter()
    with ctx.Pool(cores) as pool:
        res = pool.map(_ref_worker, jobs)
    wall = time.perf_counter() - t0
    inner = max(r[0] for r in res)      # slowest worker's scoring time (excludes import/setup)
    return cores * pts_per_core / inner, inner, wall


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import build_ref
    kind = "reference" if build_ref.built() else "port"
    cores = os.cpu_count() or 1
    pts = 1500
    if kind == "port":
        raise SystemExit("oracle/_ref is not built; run oracle/build_ref.py where /root/reference exists")
    for _ in range(min(args.warmup, 1)):
        reference_pass(cores, 200)
    vals, times = [], []
    for _ in range(args.steps):
        v, inner, _ = reference_pass(cores, pts)
        vals.append(v)
        times.append(inner)
    v = float(np.mean(vals))
    sample = "%d forked processes x %d contiguous points of the 10^6 grid (ns=64), OPENBLAS_NUM_THREADS=1" % (cores, pts)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": float(np.mean(times)) * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "C2: 1-D BQ, ns=64, expected_Z_var over a 10^6-point grid (bounded sample per step)"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------ CUDA arm
def bind_cores(world, local):
    """One process per GPU: give every rank its own slice of the host cores (the staging / zero-copy threads and the
    interpreter of eight ranks otherwise float over the same cores of one NUMA node)."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        per = len(cores) // world
        if world > 1 and per >= 1:
            os.sched_setaffinity(0, cores[local * per:(local + 1) * per])
            return len(cores), per
        return len(cores), len(cores)
    except (AttributeError, OSError):
        return os.cpu_count() or 1, 0


def ncu_pipes():
    """DMMA / FP64 pipe-busy percentages of the bench kernel from the committed ncu capture of this round
    (profiles/ncu_score_r02.json, written by profiles/summarize.py); None when absent."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_score_r02.json")) as fh:
            return json.load(fh)
    except Exception:
        return None


def max_over_ranks(v, dev, world):
    import torch
    import torch.distributed as dist
    t = torch.tensor([float(v)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def measure_pcie(world, dev, mb=64, reps=12):
    """What the platform gives for the e2e traffic pattern: every rank copies `mb` MB page-locked host -> device and device ->
    page-locked host AT THE SAME TIME (two streams), all ranks concurrently.  Returns the aggregate GB/s over the ranks (both
    directions summed) and this rank's share; 16 bytes cross PCIe per evaluation of the e2e path (8 in, 8 out)."""
    import torch
    import torch.distributed as dist
    n = mb * (1 << 20) // 8
    h_in = torch.empty(n, dtype=torch.float64).pin_memory()
    h_out = torch.empty(n, dtype=torch.float64).pin_memory()
    d_in = torch.empty(n, dtype=torch.float64, device=dev)
    d_out = torch.ones(n, dtype=torch.float64, device=dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    def burst():
        with torch.cuda.stream(s1):
            d_in.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s2):
            h_out.copy_(d_out, non_blocking=True)
    for _ in range(2):
        burst()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        burst()
    torch.cuda.synchronize()
    mine = 2 * n * 8 * reps / (time.perf_counter() - t0) * 1e-9
    t = torch.tensor([mine], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return {"aggregate_gbs_both_directions": float(t.item()), "rank0_gbs_both_directions": mine, "mb_per_copy": mb,
            "pattern": "H2D and D2H copies of page-locked buffers running concurrently on every rank"}


def cfg_c3_strong(world, rank, dev, steps=10):
    """BASELINE configs[2]: ns = 256, 10^7 query points FIXED, block-cyclic shards over the ranks, (min, first index) of the
    expected variance exchanged by the reduction kernel.  Strong scaling.  Checked against rank 0 scoring all 10^7 points."""
    import torch
    import torch.distributed as dist
    from bayesian_quadrature_b200 import BQ, GaussianKernel, synthetic
    from bayesian_quadrature_b200 import dist as bqdist
    ns, na, blk = 256, 10 ** 7, 10 ** 4
    bq = synthetic.make_bq(BQ, GaussianKernel, ns)
    bq.device = dev.index
    batch = bq._device_model().batch
    x = synthetic.query_grid(ns, na)
    x_d = torch.from_numpy(bqdist.cyclic_shard(x, world, rank, blk)).to(dev)
    esm, ev = torch.empty_like(x_d), torch.empty_like(x_d)
    ex = bqdist.PairExchange.create(dev)
    if ex is None:
        return {"skipped": "symmetric memory unavailable"}
    for _ in range(3):
        got = ex.step(batch, x_d, esm, ev, 0, cyclic_block=blk)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        ex.step_async(batch, x_d, esm, ev, 0, cyclic_block=blk)
    e1.record()
    got = ex.result()
    torch.cuda.synchronize()
    ms = max_over_ranks(e0.elapsed_time(e1) / steps, dev, world)
    out = {"workload": "C3: ns=256, 10^7 points fixed, block-cyclic shards of %d" % blk, "scaling": "strong", "n_gpus": world,
           "ms_per_step": ms, "evals_per_s": na / (ms * 1e-3), "argmin": {"min": got[0], "index": got[1]}}
    if rank == 0:                                       # single-GPU answer over ALL points (outside the timed region)
        x_full = torch.from_numpy(x).to(dev)
        e_f, v_f = torch.empty_like(x_full), torch.empty_like(x_full)
        pair = torch.empty(2, dtype=torch.float64, device=dev)
        batch.choose_step_device(x_full, e_f, v_f, pair)
        p = pair.cpu().numpy()
        out["argmin_check"] = bool(p[0] == got[0] and int(p[1]) == got[1])
        out["argmin_single_gpu"] = {"min": float(p[0]), "index": int(p[1])}
    return out


def cfg_c4_samples(world, rank, dev, steps=3):
    """BASELINE configs[3]: 1024 hyper-parameter sets x 10^5 points, the SAMPLES sharded across the ranks: every rank sets
    up and scores its 1024 / N sets chunk by chunk, accumulating the sum of -esm in sample order; the partial sums are
    all-reduced (the path's one real exchange: 10^5 doubles), divided by 1024, and reduced to (min, first index)."""
    import torch
    import torch.distributed as dist
    from bayesian_quadrature_b200 import BQ, GaussianKernel, _lib, synthetic
    from bayesian_quadrature_b200 import dist as bqdist
    ns, na, n_hyper = 64, 10 ** 5, 1024
    bq = synthetic.make_bq(BQ, GaussianKernel, ns)
    lo, hi = bqdist.shard_bounds(n_hyper, world, rank)
    n = hi - lo
    hyp4 = synthetic.hyper_sets(n_hyper)[lo:hi]
    hyp = np.zeros((n, 6))
    hyp[:, 0], hyp[:, 1], hyp[:, 3], hyp[:, 4] = hyp4.T
    opt = synthetic.options(ns)
    prior = np.tile([opt["x_mean"], opt["x_var"], opt["candidate_thresh"]], (n, 1))
    batch = _lib.Batch(n, ns, device=dev.index)
    t0 = time.perf_counter()
    info = batch.setup(np.full(n, ns), np.full(n, bq.nc), np.tile(bq.x_s, (n, 1)), np.tile(bq.l_s, (n, 1)),
                       np.tile(bq.x_c, (n, 1)), hyp, prior, check_max=True)
    setup_ms = (time.perf_counter() - t0) * 1e3
    assert (info["status"] == 0).all()
    x_d = torch.from_numpy(synthetic.query_grid(ns, na)).to(dev)
    chunk = min(n, 74)                                # 74 instances x 4 CTAs = 296 = 148 SMs x 2: one full wave per launch
    esm = torch.empty(chunk, na, dtype=torch.float64, device=dev)
    total = torch.empty(na, dtype=torch.float64, device=dev)
    pair = torch.empty(2, dtype=torch.float64, device=dev)

    def step():
        total.zero_()
        for i0 in range(0, n, chunk):
            cnt = min(chunk, n - i0)
            batch.score_device_range(i0, cnt, x_d, esm)
            batch.sum_neg_accum_device(esm, cnt, total)
        loss = bqdist.all_reduce_loss(total, n_hyper)             # NCCL all-reduce (sum) of 10^5 doubles, then / 1024
        batch.argmin_pair_device(loss, 0, pair)
        return loss
    for _ in range(2):
        loss = step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    torch.cuda.synchronize()
    ms = max_over_ranks(e0.elapsed_time(e1) / steps, dev, world)
    p = pair.cpu().numpy()
    lsum = float(loss.sum().item())
    batch.close()
    return {"workload": "C4: 1024 hyper sets x 10^5 points (ns=64), samples sharded, all-reduce of the partial loss",
            "scaling": "strong", "n_gpus": world, "ms_per_step": ms, "evals_per_s": n_hyper * na / (ms * 1e-3),
            "setup_ms": max_over_ranks(setup_ms, dev, world), "score_buffer_mb": chunk * na * 8 / 1e6,
            "argmin": {"min": float(p[0]), "index": int(p[1])}, "loss_checksum": lsum}


def cfg_c5_problems(world, rank, dev, rounds=20):
    """BASELINE configs[4]: 16384 independent problems (ns = 128 at the start), 20 rounds of score -> per-problem argmin ->
    add_observation -> candidate redraw -> re-initialisation, device resident; problems sharded across the ranks, no
    collective.  The likelihood at the chosen points is the caller's black box (numpy on the host)."""
    import torch
    import torch.distributed as dist
    from bayesian_quadrature_b200 import BatchBQ, synthetic
    from bayesian_quadrature_b200 import dist as bqdist
    n_prob, ns, na = 16384, 128, 4096
    lo, hi = bqdist.shard_bounds(n_prob, world, rank)
    P = hi - lo
    opt = synthetic.options(ns)
    x0, _ = synthetic.observations(ns)
    shifts = np.array([synthetic.problem_shift(p) for p in range(lo, hi)])
    sp = synthetic.span(ns)

    def lik(x, sh):
        npdf = lambda x, m, s: np.exp(-0.5 * ((x - m) / s) ** 2) / (np.sqrt(2 * np.pi) * s)
        return (0.5 * npdf(x, (-0.3 + sh[:, 0]) * sp, 0.16 * sp) + 0.3 * npdf(x, (0.4 + sh[:, 1]) * sp, 0.10 * sp)
                + 0.2 * npdf(x, (0.1 + sh[:, 2]) * sp, 0.3 * sp))
    l0 = np.stack([lik(np.full(P, x), shifts) for x in x0], axis=1)
    bb = BatchBQ(np.tile(x0, (P, 1)), l0, synthetic.PARAMS_TL, synthetic.PARAMS_L, opt["n_candidate"], opt["candidate_thresh"],
                 opt["x_mean"], opt["x_var"], seed=synthetic.SEED + lo, ns_reserve=rounds, device=dev.index, device_resident=True)
    grid = torch.from_numpy(synthetic.query_grid(ns, na)).to(dev)
    # warm-up outside the timed loop, on a small batch of its own: two rounds load the kernels of this capacity class
    # (CUDA loads a kernel at its first launch; ~50 ms per process that would otherwise be billed to round 0 and does
    # not shrink with the number of ranks)
    Pw = min(P, 32)
    warm = BatchBQ(np.tile(x0, (Pw, 1)), l0[:Pw], synthetic.PARAMS_TL, synthetic.PARAMS_L, opt["n_candidate"], opt["candidate_thresh"],
                   opt["x_mean"], opt["x_var"], seed=synthetic.SEED + lo, ns_reserve=rounds, device=dev.index, device_resident=True)
    for _ in range(2):
        _, xw = warm.choose_next(grid, on_device=True)
        warm.add_observations(xw, torch.from_numpy(lik(xw.cpu().numpy(), shifts[:Pw])).to(dev))
    warm.close()
    score_ms = []
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_all = time.perf_counter()
    for r in range(rounds):
        e0.record()
        idx, x_next = bb.choose_next(grid, on_device=True)
        e1.record()
        xn = x_next.cpu().numpy()                                  # (synchronises: the chosen points go to the likelihood)
        score_ms.append(e0.elapsed_time(e1))
        bb.add_observations(x_next, torch.from_numpy(lik(xn, shifts)).to(dev))
    torch.cuda.synchronize()
    total_s = max_over_ranks(time.perf_counter() - t_all, dev, world)
    score = max_over_ranks(float(np.sum(score_ms)), dev, world)
    bb.sync_host()
    out = {"workload": "C5: 16384 problems x 4096 points, ns 128 -> %d..%d, %d device-resident rounds, problems sharded, no collective"
                       % (int(bb.ns.min()), int(bb.ns.max()), rounds),
           "scaling": "strong", "n_gpus": world, "rounds": rounds, "total_s": total_s, "ms_per_step": total_s * 1e3 / rounds,
           "evals_per_s": n_prob * na * rounds / total_s, "scoring_ms_per_round": score / rounds,
           "evals_per_s_scoring_only": n_prob * na * rounds / (score * 1e-3), "timing": "host wall clock around the loop (it contains "
           "the caller's host likelihood), max over ranks; scoring_ms_per_round from CUDA events; kernels loaded by a 32-problem warm-up batch",
           "Z_mean_first_problem_of_rank0": float(bb.Z_mean()[0])}
    bb.close()
    return out


def dump_outputs(path, arrays):
    """Writes `arrays` as <path>/<name>.npy (float64).  The inputs are seeded, so two builds run with the same arguments can
    be compared output for output."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))


def run_cuda(args):
    import torch
    import torch.distributed as dist
    from bayesian_quadrature_b200 import synthetic, _lib
    from bayesian_quadrature_b200 import dist as bqdist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (this path has no CPU fallback)")
    # ONE JSON line on stdout: whatever libraries print while the run lasts (NCCL's version banner) goes to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    host_cores, cores_per_rank = bind_cores(world, local)
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    bq = build_problem()
    bq.device = local
    nc = bq.nc
    na_total = NA * world
    grid = synthetic.query_grid(NS, na_total)
    # block-cyclic shards (blocks of CYC points dealt round-robin): every rank sees the same mix of near- and far-field
    # points; with contiguous shards the ranks holding the observed region would do several times the work of the others
    CYC = 10000
    shard = bqdist.cyclic_shard(grid, world, rank, CYC) if os.environ.get("BQB_SHARD", "cyclic") == "cyclic" else grid[rank * NA:(rank + 1) * NA]
    cyc = CYC if os.environ.get("BQB_SHARD", "cyclic") == "cyclic" else 0

    # ---- setup (amortised over the grid, timed separately): wall time of a full device-model rebuild
    # (buffer allocation + uploads + setup kernel + header read-back) and of a refresh under new hyper-parameters on the
    # resident buffers (what one log-density evaluation of the sampler costs)
    bq._device_model()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    bq._invalidate_device()
    model = bq._device_model()
    torch.cuda.synchronize()
    setup_ms = (time.perf_counter() - t0) * 1e3
    p_tl, p_l = bq.gp_log_l.params, bq.gp_l.params
    rehyper = []
    for k in range(6):
        ptl = p_tl.copy(); ptl[1] = 2.0 + 0.01 * (k + 1)
        t0 = time.perf_counter()
        bq._refresh_device(ptl, p_l, check_max=True)
        rehyper.append((time.perf_counter() - t0) * 1e3)
    model = bq._device_model()
    batch = model.batch

    x_d = torch.from_numpy(shard).to(dev)
    esm = torch.empty(1, NA, dtype=torch.float64, device=dev)
    em = torch.empty(1, NA, dtype=torch.float64, device=dev)
    st = torch.empty(1, NA, dtype=torch.int32, device=dev)
    evv = torch.empty(NA, dtype=torch.float64, device=dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # 256 MiB > 126 MB L2
    pair = torch.empty(2, dtype=torch.float64, device=dev)
    pairs = torch.empty(world, 2, dtype=torch.float64, device=dev) if world > 1 else None

    # cross-rank exchange inside the reduction kernel (peer-mapped symmetric memory over NVLink); NCCL all-gather otherwise
    exch = None if os.environ.get("BQB_EXCHANGE", "p2p") == "nccl" else bqdist.PairExchange.create(dev)

    def step():
        # esm (bq.py:379-402), expected variance (bq.py:374-377) and the (min, first global index) over all shards:
        # the scoring kernel with its fused epilogue + one tiny reduce-and-exchange launch; result in page-locked memory
        if exch is not None:
            return exch.step(batch, x_d, esm[0], evv, rank * NA, cyclic_block=cyc)
        batch.choose_step_device(x_d, esm, evv, pair, offset=0 if cyc else rank * NA)
        if cyc:                                                    # local -> global index of a block-cyclic shard
            i = pair[1]
            pair[1] = (torch.floor(i / cyc) * world + rank) * cyc + torch.remainder(i, cyc)
        if world > 1:
            dist.all_gather_into_tensor(pairs.view(-1), pair)      # the path's only collective: W pairs of 16 B
            return bqdist.combine_argmin(pairs.cpu().numpy())
        p = pair.cpu().numpy()                                     # the step's device->host read (16 B)
        return float(p[0]), int(p[1])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    # clocks are sampled from here (kernel-only loops of the same kernel + the timed steps: the K timed steps alone last
    # ~6 ms at N = 1, less than one nvidia-smi sample)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    # ---- kernel-only timing of the dominant kernel (CUDA events on the launching stream)
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kern_ms = []
    for _ in range(max(args.steps, 5)):
        flush.zero_()
        k0.record()
        batch.score_device(x_d, esm, em, st)
        k1.record()
        torch.cuda.synchronize()
        kern_ms.append(k0.elapsed_time(k1))
    kern_ms_avg = float(np.mean(kern_ms))
    # executed work of one launch (device counter of DMMA instructions), and the same launch with the band skipping
    # switched off (cut-off = inf: the dense border-update algorithm SURVEY §8(d)'s W_flop counts)
    batch.work_counter(True)
    batch.score_device(x_d, esm, em, st)
    torch.cuda.synchronize()
    dmma_per_launch = batch.work_counter(False)
    batch.set_cutoff(float("inf"))
    dense_ms = []
    for _ in range(max(args.steps, 5)):
        flush.zero_()
        k0.record()
        batch.score_device(x_d, esm, em, st)
        k1.record()
        torch.cuda.synchronize()
        dense_ms.append(k0.elapsed_time(k1))
    dense_ms_avg = float(np.mean(dense_ms[1:]))
    batch.set_cutoff(72.0)

    # ---- timed region: exactly K steps, L2 flushed between steps (outside the per-step events)
    launches0 = batch.launch_count
    step_ms = []
    l2_note = "flushed between timed steps (256 MiB memset)"
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    result = None
    NSETS = 8
    sets = None
    if exch is not None:
        # the K steps are enqueued back to back; the ranks stay in step on the device through the exchange kernel, so no
        # host wake-up jitter is billed to a step.  Cold L2 without a flush kernel in the loop (its run-to-run jitter would
        # leak into the other ranks' steps through the exchange): NSETS rotating sets of input / output vectors, 24 MB
        # each, 192 MB > 126 MB of L2 in total.
        sets = [(x_d.clone(), torch.empty_like(esm[0]), torch.empty_like(evv)) for _ in range(NSETS)]
        flush.zero_()
        barrier()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for k, (s0, s1) in enumerate(evs):
            xs_k, esm_k, ev_k = sets[k % NSETS]
            s0.record()
            exch.step_async(batch, xs_k, esm_k, ev_k, rank * NA, cyclic_block=cyc)
            s1.record()
        result = exch.result()
        step_ms = [s0.elapsed_time(s1) for s0, s1 in evs]
        l2_note = "%d rotating input/output sets (%d MiB > 126 MB L2), no flush inside the timed loop" % (NSETS, NSETS * 24)
    else:
        for _ in range(args.steps):
            flush.zero_()
            torch.cuda.synchronize()
            e0.record()
            result = step()
            e1.record()
            torch.cuda.synchronize()
            step_ms.append(e0.elapsed_time(e1))
    barrier()
    launches = batch.launch_count - launches0
    ms_per_step = max_over_ranks(float(np.sum(step_ms)), dev, world) / args.steps
    if args.dump_outputs and rank == 0:
        # what the last timed step handed its caller (rank 0's shard, 16 MB, and the global pair), before the sustained loop
        # reuses the buffers
        last_esm, last_ev = (sets[(args.steps - 1) % NSETS][1:] if sets is not None else (esm[0], evv))
        dump_outputs(args.dump_outputs, {"esm": last_esm.cpu().numpy(), "expected_Z_var": last_ev.cpu().numpy(),
                                         "argmin": np.array(result, dtype=np.float64)})
    value = na_total / (ms_per_step * 1e-3)
    clocks = sampler.stop() if sampler else None

    # ---- correctness of the cross-rank exchange (outside the timed region): rank 0 scores the WHOLE N x 10^6 grid on its
    # own GPU; the exchanged (min, first global index) must be that, and no rank may have timed out in the exchange kernel
    # (PairExchange.result raises on the time-out flag out[2])
    argmin_check = None
    if world > 1 and rank == 0:
        x_full = torch.from_numpy(grid).to(dev)
        e_f, v_f = torch.empty_like(x_full), torch.empty_like(x_full)
        batch.choose_step_device(x_full, e_f, v_f, pair)
        p = pair.cpu().numpy()
        argmin_check = bool(p[0] == result[0] and int(p[1]) == result[1])
        del x_full, e_f, v_f

    # ---- sustained: >= 2 s of back-to-back steps (same rotating sets) with a clock record of its own
    sustained = None
    if not args.no_sustained:
        s_sampler = ClockSampler(local) if rank == 0 else None
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n_sus, t_sus = 0, 0.0
        if sets is None:
            sets = [(x_d.clone(), torch.empty_like(esm[0]), torch.empty_like(evv)) for _ in range(NSETS)]
        per_burst = 1000
        while t_sus < 2000.0:
            s0.record()
            for k in range(per_burst):
                xs_k, esm_k, ev_k = sets[k % NSETS]
                if exch is not None:
                    exch.step_async(batch, xs_k, esm_k, ev_k, rank * NA, cyclic_block=cyc)
                else:
                    batch.choose_step_device(xs_k, esm_k, ev_k, pair, offset=0)
            s1.record()
            if exch is not None:
                exch.result()
            torch.cuda.synchronize()
            t_sus += s0.elapsed_time(s1)
            n_sus += per_burst
        t_sus = max_over_ranks(t_sus, dev, world)
        sus_clocks = s_sampler.stop() if s_sampler else None
        sustained = {"steps": n_sus, "seconds": t_sus * 1e-3, "ms_per_step": t_sus / n_sus, "evals_per_s": na_total * n_sus / (t_sus * 1e-3),
                     "clocks": sus_clocks}
        barrier()

    if clocks is not None and not clocks.get("sm_mhz") and sustained and sustained.get("clocks"):
        clocks = dict(sustained["clocks"], source="sustained loop (no nvidia-smi sample fell inside the timed steps)")

    # ---- end to end through the public host API (BQ.expected_Z_var): numpy in, numpy out, H2D + D2H inside the timed region
    def time_e2e(x_host, reps):
        keep = [bq.expected_Z_var(x_host) for _ in range(3)]     # steady state: the caller still holds the previous result
        del keep
        barrier()
        ts = []
        for _ in range(reps):
            flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            bq.expected_Z_var(x_host)
            ts.append((time.perf_counter() - t0) * 1e3)
        barrier()
        return na_total / (max_over_ranks(float(np.sum(ts)), dev, world) / reps * 1e-3)
    x_pin = torch.from_numpy(shard).pin_memory()
    e2e_value = time_e2e(x_pin.numpy(), args.steps)               # page-locked input: the kernel reads / writes host memory in place
    d2h_bytes = bq._last_d2h_bytes
    batch.set_zero_copy(False)
    e2e_staged = time_e2e(x_pin.numpy(), max(args.steps // 2, 3))  # page-locked input, staged asynchronous copies
    batch.set_zero_copy(True)
    e2e_pageable = time_e2e(np.array(shard), max(args.steps // 2, 3))   # what a caller with a plain numpy array gets
    pcie = measure_pcie(world, dev)

    extra = {}
    if not args.no_configs:
        for name, fn in (("c3_strong", cfg_c3_strong), ("c4_samples", cfg_c4_samples), ("c5_problems", cfg_c5_problems)):
            barrier()
            try:
                extra[name] = fn(world, rank, dev)
            except Exception as e:                                 # noqa: BLE001 -- a failed extra must not take the headline with it
                extra[name] = {"error": "%s: %s" % (type(e).__name__, e)}
            torch.cuda.empty_cache()

    if rank == 0:
        peak, peak_src = fp64_peak_tflops()
        wf = w_flop(NS, nc)
        algorithmic = wf * NA / (kern_ms_avg * 1e-3) * 1e-12
        executed = dmma_per_launch * 512 / (kern_ms_avg * 1e-3) * 1e-12
        dense = wf * NA / (dense_ms_avg * 1e-3) * 1e-12
        pipes = ncu_pipes()
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "C2: 1-D BQ, ns=%d nc=%d, expected_Z_var over a 10^6-point grid per GPU (%d points total)"
                                   % (NS, nc, na_total),
                       "l2": l2_note, "parallelism": "x_a sharded, %d rank(s), %s" % (world, "block-cyclic shards of %d points" % CYC if cyc else "contiguous shards"),
                       "exchange": "p2p stores from the reduction kernel (symmetric memory)" if exch is not None else "nccl all-gather",
                       "host_cores": host_cores, "cores_per_rank": cores_per_rank},
            "roofline": {"bound": "tensor", "pipe": "FP64 DMMA (mma.m8n8k4.f64; shares the FP64 datapath with DFMA)",
                         "kernel": "bq_score_kernel<KS=16,NT=2,WARPS=8,MINB=2,STREAM=0,TABN=2048,ALIGN=1>",
                         "dmma_pipe_pct": (pipes or {}).get("dmma_pipe_pct"), "fp64_pipe_pct": (pipes or {}).get("fp64_pipe_pct"),
                         "achieved": executed, "peak": peak, "unit": "TFLOP/s", "frac": executed / peak,
                         "traffic": ncu_traffic(), "traffic_unit": "bytes per launch (ncu dram read + write)", "peak_source": peak_src,
                         "note": "achieved / frac = EXECUTED DMMA flops (device counter, 512 flop per DMMA.8x8x4) / kernel time: the pipe "
                                 "fraction.  algorithmic_* = SURVEY 8(d)'s dense border-update count W_flop / kernel time, an equivalent "
                                 "rate: the kernel skips cross-kernel blocks below e^-72 of each point's leading element (band skipping, "
                                 "DESIGN.md 4.1) and so executes fewer flops than that count.  dense_* = the same kernel with the cut-off "
                                 "at infinity.  pipe_busy_pct: ncu, sm__pipe_tensor_subpipe_dmma / sm__pipe_fp64 cycles active.",
                         "flop_per_eval": wf, "exp_per_eval": w_exp(NS, nc), "kernel_ms": kern_ms_avg,
                         "executed_dmma_per_launch": dmma_per_launch, "executed_tflops": executed, "executed_frac": executed / peak,
                         "algorithmic_achieved": algorithmic, "algorithmic_frac": algorithmic / peak,
                         "dense_kernel_ms": dense_ms_avg, "dense_tflops": dense, "dense_frac": dense / peak,
                         "pipe_busy_pct": pipes,
                         "hbm_bytes_per_eval": 28, "hbm_gbs": 28 * NA / (kern_ms_avg * 1e-3) * 1e-9},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 8 * NA, "d2h_bytes_per_step": d2h_bytes,
                    "input": "page-locked numpy array, read and written in place by the kernel over PCIe (zero copy)",
                    "pinned_staged_copies": e2e_staged, "pageable_input": e2e_pageable,
                    "pcie": pcie, "pcie_gbs_used": 16 * e2e_value * 1e-9,
                    "frac_of_pcie": 16 * e2e_value * 1e-9 / pcie["aggregate_gbs_both_directions"]},
            "gpu_launches": int(launches), "setup_ms": setup_ms, "rehyper_ms": float(np.median(rehyper)),
            "clocks": clocks, "argmin": {"min": result[0], "index": result[1]}, "argmin_check": argmin_check,
            "sustained": sustained, "configs": extra,
        }
        if world == 1 and not args.no_cpu_baseline:
            from oracle import build_ref
            if build_ref.built():
                cores = os.cpu_count() or 1
                pts = args.cpu_points
                v, inner, wall = reference_pass(cores, pts)
                v1, inner1, wall1 = reference_pass(1, 12000)
                line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "reference",
                                        "sample": "%d forked processes x %d contiguous points of the 10^6 grid, %.1f s (%.1f s scoring)"
                                                  % (cores, pts, wall, inner),
                                        "single_process_value": v1,
                                        "single_process_sample": "1 process, OPENBLAS_NUM_THREADS=1, 12000 points, %.1f s" % wall1}
            else:
                line["cpu_baseline"] = None
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the C3 / C4 / C5 sharded configurations")
    ap.add_argument("--no-sustained", action="store_true", help="skip the >= 2 s sustained loop")
    ap.add_argument("--cpu-points", type=int, default=40000,
                    help="points per host core of the cpu_baseline sample (default: ~10 s of CPU work per core)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (esm and expected variance of every point "
                         "of rank 0's grid, the (min, index) pair) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    return run_cuda(args)


if __name__ == "__main__":
    sys.exit(main())
