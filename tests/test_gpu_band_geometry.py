"""The tensor-core scoring kernels over the band geometries of tests/band_model.py: every capacity class, uniform and
clustered observations, length scales from a fraction of the spacing to several tiles of k-steps, and query vectors
whose warps span 0.02 to 128 observation spacings.  Each case is scored at lengths derived from the device's SM count,
so that whole super-tiles (nsub = 4) and every remainder of 1-3 units per CTA occur.

Per case and length: (1) a subsample with points of every (pass, path, NP or window count, nsub) cell the model reports,
and all special points, against the CPU oracle; (2) the full vector against the dense cut-off; (3) in the large classes,
against every warp forced down the wide path and against the absolute-tile kernels (BQB_REL=0); (4) the work counter
equal to the host model's prediction, exactly, with the cut-off at 72 and at infinity.  (4) is what ties the model's
coverage and conservativeness claims (tests/test_band_model.py) to the masks the kernel builds: an error that moves a
band edge by a k-step changes no result, only the counter."""
import numpy as np
import pytest

import band_model as bm
from conftest import assert_close

pytestmark = pytest.mark.gpu

CASES = bm.all_cases()


@pytest.fixture(scope="module")
def lib():
    from bayesian_quadrature_b200 import _lib
    _lib.load()
    assert _lib.device_count() >= 1
    return _lib


@pytest.fixture(scope="module")
def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _gram(x, h, w):
    return h * h * np.exp(-0.5 * (x[:, None] - x[None, :]) ** 2 / (w * w))


def subsample(g, x, case, rs):
    """Indices into x: up to four warps of every cell the model reports, the first and last valid lane of each (8 points
    per cell where the cell has four warps), plus every special point."""
    keys = []
    for ph in (0, 1):
        if g.cfg.rel:
            b = g.band(ph)
            path = np.where(b["wide"], 1, 0)
            sub = np.where(b["wide"], b["nwin"], b["NP"] * 2 + b["rect"])
        else:
            q = g.groups(ph)
            path, sub = np.zeros_like(q["width"]), q["width"]
        keys.append(np.stack([np.full(path.size, ph), path, sub, g.tiles["nsub"]], axis=1))
    idx, cells = set(), 0
    for key in keys:
        for cell in np.unique(key, axis=0):
            warps = np.nonzero((key == cell).all(axis=1) & g.valid.any(axis=1))[0]
            if warps.size == 0:
                continue
            cells += 1
            for wi in rs.choice(warps, min(4, warps.size), replace=False):
                lanes = np.nonzero(g.valid[wi])[0]
                idx.update((int(g.idx[wi, lanes[0]]), int(g.idx[wi, lanes[-1]])))
    sp = bm.special_points(case)
    q = bm.query_vector(case)
    idx.update(range(q.size - sp.size, q.size))
    return np.array(sorted(idx)), cells


def score(b, x, cut, rel_env, monkeypatch):
    monkeypatch.setenv("BQB_REL", rel_env[0])
    monkeypatch.setenv("BQB_FORCE_WIDE", rel_env[1])
    b.set_cutoff(cut)
    b.work_counter(True)
    esm, em, st = b.score_host(x)
    return esm[0], em[0], st[0], b.work_counter(False)


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_band_geometry(lib, oracle, sm_count, case, monkeypatch):
    ns, nc = case.x_s.size, case.x_c.size
    h_tl, w_tl, s_tl = case.params_tl
    h_l, w_l, _ = case.params_l
    x_sc = np.concatenate([case.x_s, case.x_c])
    # well conditioned, so that the parity tolerance means something
    assert np.linalg.cond(_gram(x_sc, h_l, w_l)) <= 1e6, case.name
    assert np.linalg.cond(_gram(case.x_s, h_tl, w_tl) + s_tl * s_tl * np.eye(ns)) <= 1e6, case.name
    mu, var = case.prior
    b = lib.Batch(1, ns)
    info = b.setup([ns], [nc], case.x_s[None], case.l_s[None], case.x_c[None], np.array([case.params_tl + case.params_l]),
                   np.array([[mu, var, case.thresh]]))
    assert info["status"][0] == 0
    b.set_presort(0)                                 # the segments reach the kernel in the order they were built
    m = oracle.OracleModel(case.x_s, case.l_s, case.x_c, case.params_tl, case.params_l, mu, var, case.thresh)
    rs = np.random.RandomState(ns)
    q = bm.query_vector(case)
    nsp = (ns + 7) & ~7
    large = case.cap >= 128
    for n in bm.lengths(bm.kernel_config(case.cap, nsp), sm_count):
        x = bm.fill(q, n)
        tag = "%s na=%d" % (case.name, n)
        g = bm.model_launch(case.x_s, x, nc, w_l, w_tl, case.cap, sm_count)
        esm, em, st, work = score(b, x, 72.0, ("1", "0"), monkeypatch)
        assert work == g.work(), (tag, work, g.work())
        # (1) the oracle
        sub, cells = subsample(g, x, case, rs)
        o_esm, o_em, o_st = m.esm_and_em(x[sub])
        print("%s: %d points of %d cells against the oracle" % (tag, sub.size, cells))
        bad = ~np.isfinite(x[sub])
        assert bad.any() and (st[sub][bad] == lib.ST_XA_BAD).all(), tag
        assert ((st[sub] & 3) == (o_st & 3)).all(), tag
        assert_close(esm[sub][~bad], o_esm[~bad], "esm " + tag)
        assert_close(em[sub][~bad], o_em[~bad], "em " + tag)
        ok = np.isfinite(x)                          # (invalid points: NaN in every variant, ST_XA_BAD compared below)
        # (2) the dense cut-off: every k-step below nsp relevant
        esm_d, em_d, st_d, work_d = score(b, x, float("inf"), ("1", "0"), monkeypatch)
        assert work_d == bm.model_launch(case.x_s, x, nc, w_l, w_tl, case.cap, sm_count, cut_arg=np.inf).work(), tag
        assert (st == st_d).all(), tag
        assert_close(esm_d[ok], esm[ok], "dense esm " + tag, rtol=1e-12, atol=1e-300)
        assert_close(em_d[ok], em[ok], "dense em " + tag, rtol=1e-12, atol=1e-300)
        # (3) the other kernels of the large classes
        if large:
            for env in (("1", "1"), ("0", "0")):
                esm_v, em_v, st_v, work_v = score(b, x, 72.0, env, monkeypatch)
                g_v = g if env[0] == "1" else bm.model_launch(case.x_s, x, nc, w_l, w_tl, case.cap, sm_count, rel=False)
                vtag = "%s BQB_REL=%s BQB_FORCE_WIDE=%s" % (tag, env[0], env[1])
                assert work_v == g_v.work(), (vtag, work_v, g_v.work())
                assert (st_v == st).all(), vtag
                assert_close(esm_v[ok], esm[ok], "esm " + vtag, rtol=1e-11, atol=1e-300)
                assert_close(em_v[ok], em[ok], "em " + vtag, rtol=1e-11, atol=1e-300)
    m.close()
    b.close()
