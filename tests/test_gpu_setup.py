"""The setup kernel (csrc/bq_setup2.cu) on ragged instances of every capacity class with tensor-core scoring kernels,
against the C restatement of the reference (oracle/bq_oracle.c) on the same inputs: everything the model block is used
for -- the header scalars, l_c, scores with shortcut, jitter-pattern and far-field points, and predictions."""
import numpy as np
import pytest

from conftest import ATOL, RTOL, assert_close

pytestmark = pytest.mark.gpu


def cases():
    """(cap, ns, nc, s_tl, s_l, check_max, shuffled) per instance; instances of one capacity class share a batch"""
    out = []
    for cap, sizes in ((16, (1, 2, 7, 8, 9, 15, 16)), (64, (17, 31, 40, 63, 64)), (128, (65, 100, 127, 128)),
                       (160, (129, 148, 160)), (256, (161, 200, 255, 256))):
        for k, ns in enumerate(sizes):
            out.append((cap, ns, (k * 3) % 7, 0.0, 0.0, bool(k & 1), bool(k & 2)))
        out.append((cap, sizes[-2], 3, 0.0, 0.05, True, False))       # noisy gp_l (SURVEY A.2 asymmetry)
        out.append((cap, sizes[-1], 16 if cap >= 64 else 5, 1e-3, 0.0, False, True))   # many candidates, noisy gp_log_l
    return out


def build(case, rs):
    """x_s, l_s, x_c, hyp, prior of one instance"""
    from bayesian_quadrature_b200 import synthetic
    cap, ns, nc, s_tl, s_l, check_max, shuffled = case
    x_s = 1.25 * (np.arange(ns, dtype=np.float64) - (ns - 1) / 2.0)
    l_s = synthetic.likelihood(max(ns, 9))(x_s)
    if shuffled:
        p = rs.permutation(ns)
        x_s, l_s = x_s[p], l_s[p]
    # candidates as bq.py:967-991 leaves them: at least candidate_thresh = 0.5 from every observation and from each other
    # (mid-points of random gaps of the 1.25-spaced observations, and points beyond both ends)
    xs = np.sort(x_s)
    spots = np.concatenate([xs[:-1] + 0.625, xs[:1] - 0.9 - 1.1 * np.arange(8), xs[-1:] + 0.9 + 1.1 * np.arange(8)])
    x_c = np.sort(rs.choice(spots, size=nc, replace=False)) if nc else np.zeros(0)
    opt = synthetic.options(max(ns, 9))
    hyp = np.array([15.0, 2.0, s_tl, 0.2, 1.3, s_l])
    prior = np.array([opt["x_mean"], opt["x_var"], opt["candidate_thresh"]])
    return x_s, l_s, x_c, hyp, prior


def zvar_bound(cap, x_s, x_c, hyp, z_mean):
    """Absolute bound on the Z_var difference: 1e-13, except for the instance of the 16 class with six candidates among
    seven observations.  Its Z_var (2.1e-3) is quad - beta' K_tl^-1 beta, two terms of about c_tl Z_mean^2 = 0.73, and the
    relative errors cond * eps of K_tl^-1 beta and of alpha_l (the bordered K_l: cond 4.6e4 there) carry
    (cond_tl + cond_l) eps c_tl Z_mean^2 = 7.9e-12 into it (1.8e-11 measured on a B200); it is held to ten times that."""
    if not (cap == 16 and x_s.size == 7 and x_c.size == 6):
        return 1e-13

    def gram(x, h, w, s):
        return h * h / (np.sqrt(2 * np.pi) * w) * np.exp(-0.5 * (x[:, None] - x[None, :]) ** 2 / w ** 2) + s * s * np.eye(x.size)
    cond = np.linalg.cond(gram(x_s, *hyp[:3])) + np.linalg.cond(gram(np.concatenate([x_s, x_c]), *hyp[3:]))
    c_tl = hyp[0] ** 2 / (np.sqrt(2 * np.pi) * hyp[1])
    return 10 * cond * np.finfo(np.float64).eps * c_tl * z_mean ** 2


def test_setup_kernel_vs_oracle(oracle):
    """Sorted and shuffled observations, 0 to 16 candidates, observation noise on either GP and both settings of the
    bq.py:942-947 guard.  For these instances cond(K_tl) <= 1.5e5 and cond of the bordered K_l <= 2.8e5, the range of
    the BASELINE configurations that are held to the parity tolerance against the reference."""
    from bayesian_quadrature_b200 import _lib
    rs = np.random.RandomState(1234)
    by_cap = {}
    for c in cases():
        by_cap.setdefault((c[0], c[5]), []).append(c)
    checked = 0
    for (cap, check_max), group in sorted(by_cap.items()):
        B = len(group)
        ns = np.array([g[1] for g in group], dtype=np.int32)
        nc = np.array([g[2] for g in group], dtype=np.int32)
        X, L, XC = np.zeros((B, cap)), np.ones((B, cap)), np.zeros((B, 16))
        H, P = np.zeros((B, 6)), np.zeros((B, 3))
        inputs = []
        for i, g in enumerate(group):
            x_s, l_s, x_c, hyp, prior = build(g, rs)
            X[i, :g[1]], L[i, :g[1]], XC[i, :g[2]], H[i], P[i] = x_s, l_s, x_c, hyp, prior
            inputs.append((x_s, l_s, x_c, hyp, prior))
        b = _lib.Batch(B, cap)
        info = b.setup(ns, nc, X, L, XC, H, P, check_max=check_max)
        for i, (x_s, l_s, x_c, hyp, prior) in enumerate(inputs):
            tag = "cap=%d check_max=%d ns=%d nc=%d" % (cap, check_max, ns[i], nc[i])
            assert info["status"][i] == 0, tag
            m = oracle.OracleModel(x_s, l_s, x_c, hyp[:3], hyp[3:], prior[0], prior[1], prior[2], check_max=check_max)
            assert_close(info["Z_mean"][i], m.Z_mean(), "Z_mean " + tag)
            assert_close(info["l_c"][i, :nc[i]], m.l_c, "l_c " + tag)
            # Z_var is a 6-10 digit cancellation of two O(1e-3 .. 1) terms (SURVEY 7.2): absolute tolerance
            assert abs(info["Z_var"][i] - m.Z_var()) < zvar_bound(cap, x_s, x_c, hyp, m.Z_mean()), (tag, info["Z_var"][i], m.Z_var())
            assert abs(info["log_lh"][i] - m.log_lh()) <= RTOL * abs(m.log_lh()), (tag, info["log_lh"][i], m.log_lh())
            x_a = np.concatenate([np.linspace(x_s.min() - 3, x_s.max() + 3, 271), x_s[:5], x_s[:5] + 0.9e-4, x_c, x_c + 0.3,
                                  [x_s.min() - 100, x_s.max() + 1e4]])
            x_row = np.zeros((B, x_a.size))
            x_row[i] = x_a
            esm, em, st = b.score_host(x_row)
            o_esm, o_em, o_st = m.esm_and_em(x_a)
            assert ((st[i] & 3) == (o_st & 3)).all(), tag
            assert_close(esm[i], o_esm, "esm " + tag, rtol=RTOL, atol=ATOL)
            assert_close(em[i], o_em, "em " + tag, rtol=RTOL, atol=ATOL)
            _, v = b.predict_host(x_row)
            _, c = m.gp_log_l_mean_cov(x_a)
            assert_close(v[i], c, "v_log_l " + tag, rtol=1e-9, atol=1e-10 * np.abs(c).max())
            m.close()
            checked += 1
        b.close()
    assert checked == len(cases())


def test_setup_launch_groups_equal_single_instance_setups():
    """A batch larger than four waves whose few largest instances exceed the two-CTA limit of the setup kernel is set up in
    two launch groups through an instance list (csrc/bq_capi.cu run_setup): every instance -- small or large, wherever it
    sits in the batch -- gets exactly the model block a single-instance batch gives it."""
    from bayesian_quadrature_b200 import _lib, synthetic
    B, ns = 640, 144
    rs = np.random.RandomState(3)
    x_s, _ = synthetic.observations(ns)
    xs = np.sort(x_s)
    opt = synthetic.options(ns)
    nc = np.full(B, 2, dtype=np.int32)
    big = rs.choice(B, size=40, replace=False)
    nc[big] = 14                                                   # n = 158 > 155: the one-CTA variant for these only
    X = np.tile(x_s, (B, 1))
    L = np.stack([synthetic.likelihood(ns, synthetic.problem_shift(p))(x_s) for p in range(B)])
    spots = np.concatenate([xs[:-1] + 0.625, xs[:1] - 0.9 - 1.1 * np.arange(8), xs[-1:] + 0.9 + 1.1 * np.arange(8)])
    XC = np.zeros((B, 16))
    for p in range(B):
        XC[p, :nc[p]] = np.sort(rs.choice(spots, size=nc[p], replace=False))
    hyp = np.tile(list(synthetic.PARAMS_TL) + list(synthetic.PARAMS_L), (B, 1))
    prior = np.tile([opt["x_mean"], opt["x_var"], opt["candidate_thresh"]], (B, 1))
    b = _lib.Batch(B, ns)
    info = b.setup(np.full(B, ns, dtype=np.int32), nc, X, L, XC, hyp, prior, check_max=True)
    assert (info["status"] == 0).all()
    for p in list(big[:4]) + [0, 1, B - 1, int(big.max()) - 1 if int(big.max()) > 0 else 2]:
        b1 = _lib.Batch(1, ns)
        i1 = b1.setup([ns], [nc[p]], X[p:p + 1], L[p:p + 1], XC[p:p + 1], hyp[p:p + 1], prior[p:p + 1], check_max=True)
        m1, mp = b1.read_model(0), b.read_model(int(p))
        # (a single instance runs the 512-thread variant, the batch's small group the 256-thread one: block-wide sums are
        # combined over 16 vs 8 warps, so the last bits may differ; the large group runs the same variant: identical)
        fin = np.abs(m1) < 1e100
        scale = np.abs(m1[fin]).max()
        assert np.array_equal(fin, np.abs(mp) < 1e100)
        assert np.allclose(m1[fin], mp[fin], rtol=1e-9, atol=1e-12 * scale), (p, np.abs(m1[fin] - mp[fin]).max())
        if p in big:
            assert np.array_equal(m1, mp), p
        assert np.isclose(i1["Z_mean"][0], info["Z_mean"][p], rtol=1e-12) and np.isclose(i1["log_lh"][0], info["log_lh"][p], rtol=1e-12)
        b1.close()
    b.close()
