"""The host model of the scoring kernels' relevance masks (tests/band_model.py) on the band-geometry inputs of
tests/test_gpu_band_geometry.py, without a GPU.

* The masks are conservative: every k-step that the exact per-point criterion needs (an observation whose exponent is
  within 72 of the point's own largest) is in the mask of the point's warp (DESIGN.md 4.1, band skipping: the hull
  criterion selects more k-steps than the per-point one, never fewer).
* The inputs reach every path of the band logic on a 148-SM device: each one is asserted by name, so that an edit to
  the query vectors that drops a case fails here.

The GPU tests compare the kernel's work counter with this model's prediction, which makes both claims hold for the
masks the kernel builds."""
import numpy as np
import pytest

import band_model as bm

SM_COUNT = 148


def launches(cap, rel=True):
    """(case, geometry) of every scoring launch of the GPU tests in capacity class `cap`"""
    out = []
    for case in bm.all_cases():
        if case.cap != cap:
            continue
        q = bm.query_vector(case)
        nsp = (case.x_s.size + 7) & ~7
        for n in bm.lengths(bm.kernel_config(cap, nsp, rel), SM_COUNT):
            out.append((case, bm.model_launch(case.x_s, bm.fill(q, n), case.x_c.size, case.params_l[1], case.params_tl[1], cap,
                                              SM_COUNT, rel)))
    return out


@pytest.fixture(scope="module", params=[16, 64, 128, 160, 256])
def class_launches(request):
    return request.param, launches(request.param)


def test_query_vectors_fit_the_shortest_launch():
    for case in bm.all_cases():
        nsp = (case.x_s.size + 7) & ~7
        assert bm.query_vector(case).size <= min(bm.lengths(bm.kernel_config(case.cap, nsp), SM_COUNT)), case.name


def test_masks_are_conservative(class_launches):
    """Every k-step a point needs lies in its warp's mask, in both passes, for every warp of every launch."""
    cap, runs = class_launches
    checked = 0
    for case, g in runs:
        for ph, w in ((0, case.params_l[1]), (1, case.params_tl[1])):
            cut = bm.cut_of(w)
            mask = g.ml if ph == 0 else g.mt
            xs = case.x_s
            # vectorised per-point criterion, ties (|lhs - rhs| within 1e-9 relative) decided exactly
            for s in range(0, g.X.shape[0], 256):
                # (the kernel clamps points beyond 1e30; there the exponents overflow and no k-step carries anything)
                X, M = g.X[s:s + 256], mask[s:s + 256]
                V = g.valid[s:s + 256] & (np.abs(X) <= 1e100)
                with np.errstate(over="ignore", invalid="ignore"):
                    d2 = (X[:, :, None] - xs[None, None, :]) ** 2
                    rhs = d2.min(axis=2) + cut
                    need = d2 <= rhs[:, :, None]
                    tie = np.abs(d2 - rhs[:, :, None]) <= 1e-9 * rhs[:, :, None]
                for i, lane in zip(*np.nonzero(V & tie.any(axis=2))):
                    need[i, lane] = False
                    exact = bm.needed_ksteps(xs, g.nsp, X[i, lane], cut)
                    assert not (exact & ~M[i]).any(), (case.name, ph, X[i, lane])
                nk = np.zeros(need.shape[:2] + (g.nks,), bool)
                nk[..., :(xs.size + 3) // 4] = np.logical_or.reduceat(need, np.arange(0, xs.size, 4), axis=2)
                missing = V[:, :, None] & nk & ~M[:, None, :]
                if missing.any():
                    i, lane, k = [int(v[0]) for v in np.nonzero(missing)]
                    raise AssertionError("%s pass %d: point %r needs k-step %d, not in its warp's mask" % (case.name, ph, X[i, lane], k))
                checked += int(V.sum())
    assert checked > 100000


@pytest.mark.parametrize("cap", [128, 160, 256])
def test_band_relative_paths_are_reached(cap):
    runs = launches(cap)
    nks_max = max(g.nks for _, g in runs)
    for ph in (0, 1):
        B = [(case, g, g.band(ph)) for case, g in runs]
        tag = "class %d pass %s" % (cap, "K_tl" if ph else "K_l")
        for NP in range(1, 13):
            assert any((b["rect"] & (b["NP"] == NP)).any() for _, _, b in B), "%s: NP = %d with rectangular pairs" % (tag, NP)
        assert any((~b["wide"] & b["has"] & (b["width"] == 24)).any() for _, _, b in B), tag + ": fast band of 24 k-steps"
        assert any((b["wide"] & ~b["holes"] & (b["width"] == 25)).any() for _, _, b in B), tag + ": wide band of 25 k-steps"
        if nks_max > 32:        # class 128 (32 k-steps): a band from k-step 8 on is at most 24 wide, one window
            assert any((b["wide"] & (b["kbeg"] > 0) & (b["nwin"] >= 2)).any() for _, _, b in B), tag + ": wide, kbeg > 0, two windows"
        assert any(b["past_ks"].any() for _, _, b in B), tag + ": a wide window past KS"
        assert any((~b["wide"] & b["has"] & (b["hi"] == g.cfg.KS)).any() for _, g, b in B), tag + ": fast band touching k-step KS - 1"
        mixed = False
        for _, g, b in B:
            act = b["has"]
            key = g.tiles["cta"] * 100000 + g.tiles["it"]
            fast_keys, wide_keys = set(key[act & ~b["wide"]]), set(key[act & b["wide"]])
            mixed |= bool(fast_keys & wide_keys)
        assert mixed, tag + ": a CTA whose warps mix fast and wide paths"
    assert any((g.band(0)["has"] & ~g.band(0)["wide"] & g.band(1)["wide"]).any() for _, g in runs), \
        "class %d: K_tl wide while K_l is fast" % cap
    for n in range(1, 5):
        assert any((g.tiles["nsub"] == n).any() for _, g in runs), "class %d: nsub = %d" % (cap, n)
    if any(g.cfg.stream for _, g in runs):
        for ph in (0, 1):
            S = [g.slab(ph) for _, g in runs if g.cfg.stream]
            assert any((s["has"] & (s["frags"] <= 256)).any() for s in S), "class %d pass %d: a slab fetched whole" % (cap, ph)
            assert any((s["frags"] > 512).any() for s in S), "class %d pass %d: a slab streamed in chunks" % (cap, ph)


def test_the_streamed_classes_are_streamed():
    assert all(g.cfg.stream for case, g in launches(256))
    assert {case.x_s.size for case, g in launches(160) if g.cfg.stream} == {150, 160}
    assert not any(g.cfg.stream for _, g in launches(128))


def test_64_class_groups_are_reached():
    runs = launches(64)
    for ph in (0, 1):
        G = [g.groups(ph) for _, g in runs]
        assert any((q["has"] & (q["g0"] > 0)).any() for q in G), "pass %d: g0 > 0" % ph
        assert any((q["has"] & (q["kend"] == 16)).any() for q in G), "pass %d: kend = KS" % ph
        for w in range(1, 17):
            assert any((q["has"] & (q["width"] == w)).any() for q in G), "pass %d: band of %d k-steps" % (ph, w)


def test_work_prediction_matches_a_hand_count():
    """count_ksteps on a small mask, against the definition (pairs of k-steps, row blocks rb < nb see k < 2 rb + 2)"""
    m = np.zeros((1, 16), bool)
    m[0, [3, 4, 9]] = True
    nb = 8
    want = 0
    for rb in range(nb):
        for k in range(min(2 * rb + 2, 16)):
            want += bool(m[0, k & ~1] or m[0, k | 1])
    assert bm.count_ksteps(m, nb)[0] == want


def test_gen_masks_rounding_matches_float_conversions():
    x = np.array([1.0 + 2.0 ** -40, -1.0 - 2.0 ** -40, 0.1, -0.1, 3.0])
    up, dn = bm._f32_round(x, True), bm._f32_round(x, False)
    assert (up >= x).all() and (dn <= x).all()
    assert (up.astype(np.float32).astype(np.float64) == up).all() and (dn.astype(np.float32).astype(np.float64) == dn).all()
    assert (np.nextafter(dn.astype(np.float32), np.float32(np.inf)) >= up.astype(np.float32)).all()
    assert bm.fma_exact(1.0 + 2.0 ** -30, 1.0 + 2.0 ** -30, -1.0) == 2.0 ** -29 + 2.0 ** -60
