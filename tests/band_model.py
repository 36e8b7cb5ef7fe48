"""Host model of the relevance masks and band decisions of the tensor-core scoring kernels (csrc/bq_score.cu).

For a sorted observation vector and a query vector this reproduces, without a GPU:

* the tiling: which points each warp of each CTA owns in each super-tile (UNIT, SUB, per_inst, full, r_n, tile_u /
  tile_n of bq_score_kernel and launch_cfg2);
* gen_masks bit for bit: the clamp to +-1e30, the hull rounded outwards to float, dc rounded up to float,
  reach = dc + hw, the fma reach^2 + cut (evaluated exactly here) and the test over k < nsp;
* the per-warp decisions of the band-relative kernels (fast or wide path, NP of the rectangular loop, whether
  rectangular row-block pairs exist, the wide path's windows) and, for the streamed kernels, the CTA's slab;
* the value of the work counter (bqb_batch_work_counter), which depends on the masks alone.

The work counter ties this model to the kernel: a GPU test that finds the counter equal to the model's prediction has
shown that the kernel built exactly the masks modelled here, so what the CPU tests prove about the model's masks
(conservative, every path reached) holds for the kernel's.
"""
from dataclasses import dataclass
from fractions import Fraction

import numpy as np

CUT_ARG = 72.0
KB = 24                      # k-steps of the band-relative register tile (BK of the launches of classes 128 / 160 / 256)


@dataclass(frozen=True)
class KernelConfig:
    cap: int                 # capacity class (padded observation capacity)
    KS: int                  # k-steps of the class (cap / 4)
    NT: int                  # point tiles of 8 per warp and sub-tile
    WARPS: int
    MINB: int                # CTAs per SM of the persistent grid
    rel: bool                # band-relative register tile (fast / wide paths)
    stream: bool             # operands streamed through slab chunks

    @property
    def UNIT(self):
        return 8 * self.NT * self.WARPS

    @property
    def SUB(self):
        return 4 // self.NT


def kernel_config(cap, nsp, rel=True):
    """The instantiation bq_score.cu launches for an instance of `nsp` padded observations in class `cap` with at most
    six candidates (one dense row block: the resident variants fit wherever they are chosen below)."""
    if cap == 16:
        return KernelConfig(16, 4, 2, 8, 2, False, False)
    if cap == 64:
        return KernelConfig(64, 16, 2, 8, 2, False, False)
    KS = cap // 4
    if rel:
        # 128: resident; 160: resident while 16 warps' scratch leaves room (nb <= 16), streamed above; 256: streamed
        return KernelConfig(cap, KS, 1, 16, 1, True, cap == 256 or (cap == 160 and nsp // 8 > 16))
    # BQB_REL=0: the absolute tile (its resident / streamed choice does not change the masks and is not modelled)
    return KernelConfig(cap, KS, 1 if cap == 256 else 2, 8, 1, False, cap == 256)


def grid_ctas(cfg, na, sm_count):
    n_units = -(-na // cfg.UNIT)
    return max(1, min(sm_count * cfg.MINB, n_units))


def warp_tiles(cfg, na, sm_count):
    """One row per (CTA, super-tile, warp): arrays cta, it, warp, base (first point), npw (points), nsub (sub-tiles)."""
    UNIT, SUB = cfg.UNIT, cfg.SUB
    n_units = -(-na // UNIT)
    G = grid_ctas(cfg, na, sm_count)
    full = n_units // (G * SUB)
    R = n_units - full * G * SUB
    rows = []
    for cta in range(G):
        r_lo = full * G * SUB + (cta * R) // G
        r_n = ((cta + 1) * R) // G - (cta * R) // G
        n_it = full + (1 if r_n > 0 else 0)
        for it in range(n_it):
            tu, tn = ((it * G + cta) * SUB, SUB) if it < full else (r_lo, r_n)
            npw = 8 * cfg.NT * tn
            for w in range(cfg.WARPS):
                rows.append((cta, it, w, tu * UNIT + w * npw, npw, tn))
    a = np.array(rows, dtype=np.int64).reshape(-1, 6)
    return {k: a[:, i] for i, k in enumerate(("cta", "it", "warp", "base", "npw", "nsub"))}


def _f32_round(x, up):
    """__double2float_ru (up) / __double2float_rd of finite doubles within the float range, as doubles"""
    f = x.astype(np.float32)
    fd = f.astype(np.float64)
    fix = fd < x if up else fd > x
    f[fix] = np.nextafter(f[fix], np.float32(np.inf if up else -np.inf))
    return f.astype(np.float64)


def fma_exact(a, b, c):
    """a * b + c with one rounding (the device fma), for finite doubles; inf if c is inf"""
    if np.isinf(c):
        return float(c)
    return float(Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c)))


def cut_of(w, cut_arg=CUT_ARG):
    """cut_arg / |H_NHL|: H_NHL = -0.5 / (w * w) is what the setup kernel writes into the model header"""
    nh = -0.5 / (w * w)
    return cut_arg / abs(nh)


def gen_masks(xs_sorted, nsp, X, valid, cuts):
    """The masks gen_masks builds for warps whose points are the rows of X [n, 32] (lanes with valid = False do not count).
    xs_sorted: the ns sorted observations (padding to nsp sits at 1e150).  cuts: one cut-off per pass (K_l, K_tl).
    Returns one boolean array [n, nsp / 4] per pass: bit ks is k-step ks."""
    xs = np.full(nsp, 1e150)
    xs[:xs_sorted.size] = xs_sorted
    n = X.shape[0]
    xc = np.clip(np.where(valid, X, 0.0), -1e30, 1e30)
    lo = np.where(valid, _f32_round(xc, False), np.inf).min(axis=1)
    hi = np.where(valid, _f32_round(xc, True), -np.inf).max(axis=1)
    any_valid = valid.any(axis=1)
    lo, hi = np.where(any_valid, lo, 0.0), np.where(any_valid, hi, 0.0)
    c = 0.5 * (lo + hi)
    hw = 0.5 * (hi - lo)
    dk = np.abs(xs[None, :] - c[:, None])
    dcf = _f32_round(np.minimum(dk.min(axis=1), 3e38), True)
    reach = dcf + hw
    t = np.maximum(dk - hw[:, None], 0.0)
    t2 = t * t
    out = []
    for cut in cuts:
        r2 = np.array([fma_exact(r, r, cut) for r in reach]) if n else np.zeros(0)
        rel = (t2 <= r2[:, None]) & any_valid[:, None]
        out.append(rel.reshape(n, nsp // 4, 4).any(axis=2))
    return out


def needed_ksteps(xs_sorted, nsp, x, cut):
    """The exact per-point criterion: k-step ks is needed by point x if one of its (real) observations has an exponent
    within cut_arg of the point's own largest, i.e. d^2 <= dmin^2 + cut.  float64 with ties decided exactly."""
    d2 = (x - xs_sorted) ** 2
    rhs = d2.min() + cut
    need = d2 <= rhs
    close = np.abs(d2 - rhs) <= 1e-9 * rhs
    if close.any():
        fx, fxs = Fraction(float(x)), [Fraction(float(v)) for v in xs_sorted]
        fd2 = [(fx - v) ** 2 for v in fxs]
        frhs = min(fd2) + Fraction(float(cut))
        for k in np.nonzero(close)[0]:
            need[k] = fd2[k] <= frhs
    ks = np.zeros(nsp // 4, bool)
    ks[np.nonzero(need)[0] // 4] = True
    return ks


def count_ksteps(mask, nb):
    """count_ksteps of bq_score.cu for boolean masks [n, nks]: sum over row blocks rb < nb of the relevant k-steps below
    2 rb + 2, at pair granularity"""
    pair = mask.reshape(mask.shape[0], -1, 2).any(axis=2)
    m = np.repeat(pair, 2, axis=1)
    j = np.arange(mask.shape[1])
    weight = np.maximum(nb - j // 2, 0)
    return (m * weight[None, :]).sum(axis=1)


@dataclass
class Geometry:
    """Everything bq_score_kernel decides from the masks of one launch (one instance)."""
    cfg: KernelConfig
    nsp: int
    ndb: int
    tiles: dict
    ml: np.ndarray           # [n, nks] masks of the K_l pass per warp tile
    mt: np.ndarray           # [n, nks] K_tl
    X: np.ndarray            # [n, 32] the warp's points (0 where not valid)
    valid: np.ndarray
    idx: np.ndarray          # [n, 32] index of each lane's point in the query vector (-1: none)

    @property
    def nb(self):
        return self.nsp // 8

    @property
    def nks(self):
        return self.nsp // 4

    def work(self):
        """bqb_batch_work_counter after one launch: NT * sum over warps and sub-tiles of count_ksteps(K_l) +
        ndb popc(K_l) + count_ksteps(K_tl)"""
        per = count_ksteps(self.ml, self.nb) + self.ndb * self.ml.sum(axis=1) + count_ksteps(self.mt, self.nb)
        return int(self.cfg.NT * (per * self.tiles["nsub"]).sum())

    def band(self, ph):
        """Per-warp band decisions of pass ph (0: K_l, 1: K_tl) of the band-relative kernels, as a dict of arrays."""
        m = self.ml if ph == 0 else self.mt
        n, nks = m.shape
        has = m.any(axis=1)
        lo = np.where(has, m.argmax(axis=1), 0)
        hi = np.where(has, nks - m[:, ::-1].argmax(axis=1), 0)
        holes = has & (m.sum(axis=1) != hi - lo)
        width = hi - (lo & ~1)
        wide = has & ((width > KB) | holes)
        k0 = np.where(wide, 0, lo & ~1)
        # fast path: relative mask rm = m >> k0 has no holes and starts in group 0, so plain_band holds and the rectangular
        # loop takes NP = kend2 / 2 pairs, kend2 the band end rounded up to a pair
        kend2 = (hi - k0 + 1) & ~1
        NP = np.where(has & ~wide, kend2 >> 1, 0)
        rbx = ((k0 + kend2) >> 1) & ~1
        rect = np.zeros(n, bool)
        if self.cfg.stream:
            slab = self.slab(ph)
            for i in np.nonzero(has & ~wide)[0]:
                rb_first, R, res = slab["rb_first"][i], slab["R"][i], slab["res"][i]
                rb1s = [self.nb] if res else list(range(rb_first + R, self.nb, R)) + [self.nb]
                rb0 = rb_first
                for rb1 in rb1s:
                    rbf = min(rb1, max(rb0, rbx[i]))
                    rect[i] |= rbf + 1 < rb1
                    rb0 = rb1
        else:
            rect = has & ~wide & (np.minimum(self.nb, rbx) + 1 < self.nb)
        kbeg = np.where(wide, lo & ~7, 0)
        nwin = np.where(wide, -(-(hi - kbeg) // KB), 0)
        return {"has": has, "lo": lo, "hi": hi, "width": width, "wide": wide, "holes": holes, "k0": k0, "kend2": kend2,
                "NP": NP, "rect": rect, "kbeg": kbeg, "kend": np.where(wide, hi, 0), "nwin": nwin,
                "past_ks": wide & (kbeg + KB * nwin > self.cfg.KS)}

    def groups(self, ph):
        """g0 / kend of the jump-table loops (mask_groups of the absolute mask) and the band width hi - lo"""
        m = self.ml if ph == 0 else self.mt
        has = m.any(axis=1)
        lo = np.where(has, m.argmax(axis=1), 0)
        hi = np.where(has, m.shape[1] - m[:, ::-1].argmax(axis=1), 0)
        return {"has": has, "g0": lo >> 2, "kend": (hi + 3) & ~3, "width": hi - lo}

    def slab(self, ph):
        """make_slab_plan of the CTA's union mask of pass ph, per warp tile: rb_first, W, slab fragments, R, whole (res)"""
        m = self.ml if ph == 0 else self.mt
        key = self.tiles["cta"] * 100000 + self.tiles["it"]
        _, inv = np.unique(key, return_inverse=True)
        um = np.zeros((inv.max() + 1 if inv.size else 0, m.shape[1]), bool)
        np.logical_or.at(um, inv, m)
        um = um[inv]
        has = um.any(axis=1)
        lo = np.where(has, um.argmax(axis=1), 0)
        hi = np.where(has, um.shape[1] - um[:, ::-1].argmax(axis=1), 0)
        klo = lo & ~3
        khi = np.minimum((hi + 3) & ~3, self.nks)
        W = np.where(has, khi - klo, 0)
        rb_first = klo >> 1
        frags = (self.nb - rb_first) * W
        cap = chunk_frags(self.cfg)
        R = np.maximum(2, (cap // np.maximum(W, 1)) & ~1)
        return {"has": has, "rb_first": rb_first, "W": W, "frags": np.where(has, frags, 0), "R": R, "res": frags <= 2 * cap}


def chunk_frags(cfg):
    """chunk buffer size of the streamed band-relative launches with one dense row block (launch_cfg2: the largest multiple
    of 16 fragments <= 256 that fits); only decides whether slabs between 256 and 512 fragments are chunked"""
    return 256


def model_launch(xs_sorted, x_a, ncand, w_l, w_tl, cap, sm_count, rel=True, cut_arg=CUT_ARG):
    """The masks of one scoring launch of one instance over the query vector x_a (in the order the kernel sees it)."""
    ns = xs_sorted.size
    nsp = (ns + 7) & ~7
    cfg = kernel_config(cap, nsp, rel)
    na = x_a.size
    tiles = warp_tiles(cfg, na, sm_count)
    lane = np.arange(32)
    idx = tiles["base"][:, None] + lane[None, :]
    ok = (lane[None, :] < tiles["npw"][:, None]) & (idx < na)
    idx = np.where(ok, idx, -1)
    X = np.where(ok, x_a[np.clip(idx, 0, max(na - 1, 0))], 0.0)
    valid = ok & np.isfinite(X)
    X = np.where(valid, X, 0.0)
    ml, mt = gen_masks(xs_sorted, nsp, X, valid, (cut_of(w_l, cut_arg), cut_of(w_tl, cut_arg)))
    return Geometry(cfg, nsp, (ncand + 2 + 7) // 8, tiles, ml, mt, X, valid, idx)


# ------------------------------------------------------------------------------------------------------ the test inputs
@dataclass
class Case:
    name: str
    x_s: np.ndarray          # sorted observations
    l_s: np.ndarray
    x_c: np.ndarray
    params_tl: tuple
    params_l: tuple
    spacing: float           # typical observation spacing
    thresh: float = 0.5

    @property
    def prior(self):
        return 0.0, float(max(np.ptp(self.x_s), 2.0) ** 2 / 4)

    @property
    def cap(self):
        ns = self.x_s.size
        return next(c for c in (16, 64, 128, 160, 256) if ns <= c)


UNIFORM = {"narrow": (0.3, 0.5, 0.0), "synthetic": (1.3, 2.0, 0.0), "broad": (1.0, 6.0, 0.05)}     # (w_l, w_tl, s_tl)
SIZES = (16, 64, 100, 128, 150, 160, 256)
#: query segments: 32 consecutive points span H observation spacings
SPANS = (0.02, 0.5, 2, 8, 16, 32, 48, 64, 80, 96, 128)


def _likelihood(x):
    sp = max(np.ptp(x), 1.0)
    return np.exp(-0.5 * ((x - x.mean() - 0.1 * sp) / (0.3 * sp)) ** 2) * 0.3 + 1e-3


def _candidates(x_s, spacing, rs):
    """2 to 6 candidates, half inside the data (midway between neighbours), half beyond it"""
    n = int(rs.randint(2, 7))
    gaps = 0.5 * (x_s[1:] + x_s[:-1])
    inside = np.sort(rs.choice(gaps, n // 2, replace=False)) if x_s.size > 1 and n // 2 else np.zeros(0)
    outside = [x_s.max() + 1.1 * spacing * (1 + j) if j % 2 == 0 else x_s.min() - 1.1 * spacing * (1 + j) for j in range(n - n // 2)]
    return np.sort(np.concatenate([inside, outside]))


def make_case(ns, kind):
    rs = np.random.RandomState(1000 * ns + len(kind))
    if kind == "clustered":
        xs, x, sp = [], 0.0, 1.2
        while len(xs) < ns:
            g, step = int(rs.randint(6, 21)), rs.uniform(1.0, 1.4)
            for _ in range(min(g, ns - len(xs))):
                xs.append(x)
                x += step
            x += rs.uniform(3, 40) * sp
        x_s = np.array(xs) - 0.5 * (xs[0] + xs[-1])
        w_l, w_tl, s_tl = 0.9, 2.0, 0.05         # (noise: K_tl of groups at spacing 1.0 reaches cond 1e7 without)
    else:
        sp = 1.25
        x_s = sp * (np.arange(ns) - (ns - 1) / 2.0)
        w_l, w_tl, s_tl = UNIFORM[kind]
    h_tl = 1.0 if s_tl else 4.0
    return Case("%s-%d" % (kind, ns), x_s, _likelihood(x_s), _candidates(x_s, sp, rs), (h_tl, w_tl, s_tl), (0.3, w_l, 0.0), sp)


def all_cases():
    return [make_case(ns, kind) for ns in SIZES for kind in ("narrow", "synthetic", "broad", "clustered")]


def query_vector(case):
    """Sorted segments of constant point spacing over the domain plus 6 length scales on each side (32 consecutive points
    spanning H observation spacings; the fine ones in four pieces, at the ends and inside), a segment alternating
    between a narrow and a wide spacing every 256 points, and the special points: shortcut and near-shortcut points,
    points around the candidates, far beyond both ends and invalid ones."""
    w = max(case.params_l[1], case.params_tl[1])
    lo, hi = case.x_s.min() - 6 * w, case.x_s.max() + 6 * w
    L = hi - lo
    segs = []
    for H in SPANS:
        step = H * case.spacing / 32
        n = int(L / step) + 1
        if n <= 4096:
            segs.append(lo + step * np.arange(n))
        else:
            for start in (lo, lo + 0.3 * L, lo + 0.62 * L, hi - 1023 * step):
                segs.append(start + step * np.arange(1024))
    segs.append(np.repeat(np.linspace(lo, hi, 32)[None, :], 4, axis=0).ravel())          # whole domain per warp
    alt, x = [], lo                                                                        # one CTA, fast and wide warps
    while x < hi:
        for H in (2, 64):
            alt.append(x + H * case.spacing / 32 * np.arange(256))
            x = alt[-1][-1] + H * case.spacing / 32
    segs.append(np.concatenate(alt))
    segs.append(special_points(case))
    return np.concatenate(segs)


def special_points(case):
    xs, xc, t = case.x_s, case.x_c, case.thresh
    lo, hi = xs.min(), xs.max()
    return np.concatenate([xs, xs + 0.9e-4, xs - 0.9e-4, xs + 1.05e-4, xs - 1.05e-4, xc, xc + 0.3 * t, xc - 0.99 * t,
                           xc + 1.01 * t, [lo - 100, hi + 1e4, -1e300, 1e300, np.nan, np.inf, -np.inf]])


def lengths(cfg, sm_count):
    """Query lengths of one launch: a full round of whole super-tiles plus a remainder of r_n in {1, 2} units per CTA
    (nsub = SUB, 1, 2) and a remainder only, of r_n in {SUB - 1, SUB} (nsub = 3, 4 for SUB = 4)"""
    G = sm_count * cfg.MINB
    return [cfg.UNIT * (G * cfg.SUB + (3 * G) // 2) + 37, cfg.UNIT * ((G * (2 * cfg.SUB - 1)) // 2) + 5]


def fill(x, n):
    """x repeated cyclically to n points"""
    return np.resize(x, n)
