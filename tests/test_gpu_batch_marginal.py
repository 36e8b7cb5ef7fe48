"""BatchBQ's marginalisation over per-problem hyper-parameter samples: the batched log density, grouped scoring, the
segmented sample reduction, marginal_loss against the single-problem BQ, and choose_next(n=...)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PARAMS = ["h", "w"]


def make_batch(P=5, ns0=20, seed=31, device_resident=False, vary=True, params_tl=None):
    """P synthetic problems; with ``vary`` problem p gets P - 1 - p extra observations (the others merge), so the
    problems have different ns."""
    from bayesian_quadrature_b200 import BatchBQ, synthetic
    x0, _ = synthetic.observations(ns0)
    fl = [synthetic.likelihood(ns0, synthetic.problem_shift(p)) for p in range(P)]
    opt = synthetic.options(ns0)
    bb = BatchBQ(np.tile(x0, (P, 1)), np.stack([f(x0) for f in fl]),
                 synthetic.PARAMS_TL if params_tl is None else params_tl, synthetic.PARAMS_L,
                 opt["n_candidate"], opt["candidate_thresh"], opt["x_mean"], opt["x_var"], seed=seed, ns_reserve=8,
                 device_resident=device_resident)
    if vary:
        for r in range(P - 1):
            bb.sync_host()
            x_new = np.where(np.arange(P) <= r, x0.max() + 1.25 * (r + 1), bb.x_s[:, 0] + 0.1)
            bb.add_observations(x_new, np.array([fl[p](x_new[p]) for p in range(P)]))
    bb.sync_host()
    return bb, fl, opt


def bq_of(bb, p, opt):
    """The single-problem BQ object of problem p (same observations, candidates and hyper-parameters)."""
    from bayesian_quadrature_b200 import BQ, GaussianKernel, synthetic
    bb.sync_host()
    n, c = int(bb.ns[p]), int(bb.nc[p])
    bq = BQ(bb.x_s[p, :n].copy(), bb.l_s[p, :n].copy(), kernel=GaussianKernel, **opt)
    bq.init(params_tl=synthetic.PARAMS_TL, params_l=synthetic.PARAMS_L)
    bq.x_c, bq.nc = bb.x_c[p, :c].copy(), c
    return bq


def sample_sets(P, S, seed=5):
    from bayesian_quadrature_b200 import synthetic
    h = synthetic.hyper_sets(P * S, seed=seed).reshape(P, S, 4)
    return np.ascontiguousarray(h[..., :2]), np.ascontiguousarray(h[..., 2:])


@pytest.mark.parametrize("device_resident", [False, True])
def test_log_lh_rows_equal_single_problem_log_lh_batch(device_resident):
    import torch
    bb, _, opt = make_batch(device_resident=device_resident)
    assert len(set(bb.ns.tolist())) == bb.P
    grid = torch.from_numpy(np.linspace(-25, 25, 2001)).cuda()
    idx0, _ = bb.choose_next(grid)
    esm0 = bb._esm.clone()
    zm0, zv0 = bb.Z_mean().copy(), bb.Z_var().copy()
    htl, hl = sample_sets(bb.P, 3, seed=9)
    htl[1, 0, 1] = -1.0                                   # invalid value -> -inf
    htl[2, 1, 0] = 1e6                                    # "GP mean is too large" -> -inf
    bqs = [bq_of(bb, p, opt) for p in range(bb.P)]
    for r in range(3):
        got = bb.log_lh(htl[:, r], hl[:, r], PARAMS)
        want = np.array([bqs[p].log_lh_batch(htl[p, r][None], hl[p, r][None], PARAMS)[0] for p in range(bb.P)])
        assert (np.isfinite(got) == np.isfinite(want)).all(), (r, got, want)
        fin = np.isfinite(want)
        assert np.allclose(got[fin], want[fin], rtol=1e-9, atol=0), (r, got, want)
    assert np.isneginf(bb.log_lh(htl[:, 0], hl[:, 0], PARAMS)[1])
    assert np.isneginf(bb.log_lh(htl[:, 1], hl[:, 1], PARAMS)[2])
    # the batch's scoring model is restored exactly
    assert np.array_equal(bb.Z_mean(), zm0) and np.array_equal(bb.Z_var(), zv0)
    idx1, _ = bb.choose_next(grid)
    assert np.array_equal(idx0, idx1) and torch.equal(esm0, bb._esm)
    bb.close()


def _class_batch(ns, G, S, generic):
    """G * S instances of one ns-observation problem under G * S different hyper-parameter sets."""
    from bayesian_quadrature_b200 import _lib, synthetic
    x_s, l_s = synthetic.observations(ns)
    opt = synthetic.options(ns)
    x_c = (x_s[:-1] + 0.6)[::max(1, ns // 6)][:6]
    h = synthetic.hyper_sets(G * S, seed=ns)
    hyp = np.stack([h[:, 0], h[:, 1], np.zeros(G * S), h[:, 2], h[:, 3], np.zeros(G * S)], axis=1)
    prior = np.tile([opt["x_mean"], opt["x_var"], opt["candidate_thresh"]], (G * S, 1))
    b = _lib.Batch(G * S, _lib.ns_capacity(ns))
    if generic:
        b.set_approx(0, force_generic=True)
    info = b.setup(np.full(G * S, ns), np.full(G * S, x_c.size), np.tile(x_s, (G * S, 1)), np.tile(l_s, (G * S, 1)),
                   np.tile(x_c, (G * S, 1)), hyp, prior)
    assert (info["status"] == 0).all()
    return b, synthetic.span(ns)


@pytest.mark.parametrize("ns,generic", [(40, False), (100, False), (150, False), (200, False), (40, True)])
def test_grouped_scoring_equals_replicated_rows(ns, generic):
    import torch
    G, S, na = 3, 4, 1537
    b, sp = _class_batch(ns, G, S, generic)
    assert b.ns_max in ((64, 128, 160, 256) if not generic else (64,))
    grid = torch.from_numpy(np.stack([np.linspace(-2 * sp + g, 2 * sp - g, na) for g in range(G)])).cuda()
    rep = grid.repeat_interleave(S, dim=0).contiguous()
    want = torch.empty(G * S, na, dtype=torch.float64, device="cuda")
    b.score_device(rep, want)
    got = torch.full_like(want, np.nan)
    flags = torch.zeros(G * S, dtype=torch.int32, device="cuda")
    b.score_device_grouped(0, G * S, grid, S, got, None, None, flags)
    assert torch.equal(got, want)
    part = torch.full_like(want, np.nan)
    b.score_device_grouped(S, 2 * S, grid[1:], S, part)          # a chunk starting on the second problem
    assert torch.equal(part[:2 * S], want[S:])
    with pytest.raises(ValueError):
        b.score_device_grouped(1, S, grid, S, part)              # not on a group boundary
    with pytest.raises(ValueError):
        b.score_device_grouped(0, G * S, grid[:G - 1], S, part)  # fewer grid rows than groups
    b.close()


@pytest.mark.parametrize("na", [0, 1, 4099])
def test_segmented_reduction_matches_sum_neg_accum(na):
    import torch
    from bayesian_quadrature_b200 import _lib
    b = _lib.Batch(13, 16)                                # mean_neg_device averages the first n_inst = 13 rows
    g = torch.Generator(device="cuda").manual_seed(na)
    esm = torch.rand(16, na, dtype=torch.float64, device="cuda", generator=g) * 1e-3 - 3e-4
    start = torch.rand(3, na, dtype=torch.float64, device="cuda", generator=g)
    if na == 0:                                           # empty tensors: nothing to read or write, no error
        b.sum_neg_accum_groups_device(esm, 3, 5, start)
        b.close()
        return

    def neg_sum(acc, rows):                               # the additions of numpy's mean(axis=0), in row order
        acc = acc.clone()
        for r in rows:
            acc += -r
        return acc

    # one group of 16 rows, starting from a non-zero accumulator
    want = neg_sum(start[0], esm)
    acc = start[0].clone()
    b.sum_neg_accum_device(esm, 16, acc)
    assert torch.equal(acc, want)
    got = start[:1].clone()
    b.sum_neg_accum_groups_device(esm, 1, 16, got)
    assert torch.equal(got[0], want)
    # the mean over the batch's 13 rows: the same additions from 0, then one division (in numpy: torch divides by a
    # scalar as a multiplication with its reciprocal)
    loss = torch.full((na,), np.nan, dtype=torch.float64, device="cuda")
    b.mean_neg_device(esm, loss)
    want = neg_sum(torch.zeros(na, dtype=torch.float64, device="cuda"), esm[:13]).cpu().numpy() / 13
    assert np.array_equal(loss.cpu().numpy(), want)
    # S = 1: every row its own group
    got = start.clone()
    b.sum_neg_accum_groups_device(esm, 3, 1, got)
    assert torch.equal(got, start - esm[:3])
    # S = 5 does not divide the 16-row buffer: three groups, the last row unused
    got = start.clone()
    b.sum_neg_accum_groups_device(esm, 3, 5, got)
    for k in range(3):
        want = neg_sum(start[k], esm[5 * k:5 * k + 5])
        assert torch.equal(got[k], want), k
        acc = start[k].clone()
        b.sum_neg_accum_device(esm[5 * k:5 * k + 5], 5, acc)
        assert torch.equal(acc, want), k
    b.close()


@pytest.mark.parametrize("per_problem_grid", [False, True])
def test_marginal_loss_equals_single_problem_marginal_loss(per_problem_grid):
    import torch
    from bayesian_quadrature_b200 import _lib
    bb, _, opt = make_batch()
    P, S, na = bb.P, 4, 2049
    htl, hl = sample_sets(P, S)
    grid = np.linspace(-25, 25, na)
    x_a = np.stack([grid + 0.37 * p for p in range(P)]) if per_problem_grid else grid
    model_bytes = 8 * _lib.load().bqb_model_doubles(bb.batch._h)
    bb.MODEL_CHUNK_BYTES = 2 * S * model_bytes             # two problems per setup chunk ...
    bb.LOSS_CHUNK_BYTES = 8 * S * na                       # ... one per scoring launch
    assert bb._chunks(S, na) == (2, 1)
    got = bb.marginal_loss(x_a, htl, hl, PARAMS).cpu().numpy()
    identical = 0
    for p in range(P):
        bq = bq_of(bb, p, opt)
        loss, batch = bq.marginal_loss(x_a[p] if per_problem_grid else x_a, htl[p], hl[p], PARAMS)
        batch.close()
        want = loss.cpu().numpy()
        rel = np.abs(got[p] - want) / np.abs(want)
        assert rel.max() <= 1e-12, (p, rel.max())
        assert int(np.argmin(got[p])) == int(np.argmin(want))
        identical += int(np.array_equal(got[p], want))
    assert identical == P                                  # the same additions in the same order as BQ.marginal_loss
    # one chunk of everything gives the same rows bit for bit
    bb.MODEL_CHUNK_BYTES, bb.LOSS_CHUNK_BYTES = 1 << 30, 64 << 20
    assert torch.equal(bb.marginal_loss(x_a, htl, hl, PARAMS).cpu(), torch.from_numpy(got))
    bb.close()


def test_choose_next_marginal_host_equals_device_resident():
    import torch
    host, fl, _ = make_batch(seed=123)
    dev, _, _ = make_batch(seed=123, device_resident=True)
    grid = np.linspace(-25, 25, 1501)
    # the fixed-hyper-parameter path: launches counted before any marginal call
    c0 = host.batch.launch_count
    idx_plain, _ = host.choose_next(grid)
    plain_launches = host.batch.launch_count - c0
    esm_plain = host._esm.clone()
    for rnd in range(3):
        zm, zv = host.Z_mean().copy(), host.Z_var().copy()
        idx_h, x_h = host.choose_next(grid, n=3, params=PARAMS)
        assert np.array_equal(host.Z_mean(), zm) and np.array_equal(host.Z_var(), zv)
        zm_d = dev.Z_mean().copy()
        idx_d, x_d = dev.choose_next(torch.from_numpy(grid).cuda(), on_device=True, n=3, params=PARAMS)
        assert np.array_equal(dev.Z_mean(), zm_d)
        assert np.array_equal(idx_d.cpu().numpy(), idx_h) and np.array_equal(x_d.cpu().numpy(), x_h), rnd
        if rnd == 0:
            c0 = host.batch.launch_count
            idx_again, _ = host.choose_next(grid)
            assert host.batch.launch_count - c0 == plain_launches
            assert np.array_equal(idx_again, idx_plain) and torch.equal(host._esm, esm_plain)
        l_new = np.array([fl[p](x_h[p]) for p in range(host.P)])
        host.add_observations(x_h, l_new)
        dev.add_observations(x_d, torch.from_numpy(l_new).cuda())
    host.close()
    dev.close()


def test_choose_next_with_given_hypers_is_the_argmin_of_marginal_loss():
    bb, _, _ = make_batch()
    htl, hl = sample_sets(bb.P, 2, seed=3)
    grid = np.linspace(-25, 25, 777)
    idx, x_next = bb.choose_next(grid, hypers=(htl, hl), params=PARAMS)
    loss = bb.marginal_loss(grid, htl, hl, PARAMS).cpu().numpy()
    assert np.array_equal(idx, loss.argmin(axis=1)) and np.array_equal(x_next, grid[idx])
    bb.close()


def test_device_sampler_chain_is_independent_of_the_batch():
    P, seed = 4, 1000
    bb, _, _ = make_batch(P=P, vary=False)
    htl, hl = bb.sample_hypers(PARAMS, n=3, nburn=2, seed=seed)
    assert htl.shape == (P, 3, 2) and hl.shape == (P, 3, 2)
    for i in range(3):
        assert np.isfinite(bb.log_lh(htl[:, i], hl[:, i], PARAMS)).all()
    from bayesian_quadrature_b200 import BatchBQ
    for p in (0, P - 1):
        n = int(bb.ns[p])
        single = BatchBQ(bb.x_s[p:p + 1, :n], bb.l_s[p:p + 1, :n], bb.hyp[p, :3], bb.hyp[p, 3:], bb.n_candidate, bb.thresh,
                         bb.prior[p, 0], bb.prior[p, 1], seed=31 + p, ns_reserve=8)          # make_batch's candidate stream
        assert np.array_equal(single.x_c[0], bb.x_c[p])
        s_tl, s_l = single.sample_hypers(PARAMS, n=3, nburn=2, seed=seed, first_problem=p)
        assert np.array_equal(s_tl[0], htl[p]) and np.array_equal(s_l[0], hl[p]), p
        single.close()
    bb.close()


def test_zero_probability_start_names_the_problem():
    from bayesian_quadrature_b200 import synthetic
    ptl = np.tile(synthetic.PARAMS_TL, (3, 1))
    ptl[1, 0] = 1e6                                       # problem 1 starts where the "GP mean is too large" guard fires
    bb, _, _ = make_batch(P=3, vary=False, params_tl=ptl)
    with pytest.raises(RuntimeError, match="problem 1"):
        bb.sample_hypers(PARAMS, n=1, nburn=1)
    bb.close()
