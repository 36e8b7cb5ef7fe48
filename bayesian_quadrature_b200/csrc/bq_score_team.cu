// Scoring kernel of the ns <= 64 class, second generation ("team" kernel).
//
// Same mathematics, operands and per-point tail as bq_score.cu (the bordered update of bq.py:447-527 /
// bq_c.pyx:425-535 written as V = (c L^-1) E with a generated cross-kernel tile E and band skipping); what changes is
// how the work is laid out on an SM.
//
// ncu + subtractive timing of the first-generation kernel (profiles/ncu_score_r02.md): 128 registers per thread (the
// cross-kernel tile bf[16][2] lives in registers) allow 16 warps per SM, every warp walks a long serial chain per
// 32-point super-tile (masks -> exps -> 8 row blocks of LDS -> DMMA -> ... -> tail) and the FP64 pipe idles half of the
// time: T(warps per SM) = 0.149 + 2.18 / warps ms per 10^6 points (0.422 ms at 8, 0.285 at 16) -- latency bound, with a
// pipe-bound floor of 0.15 ms.  Here
//   * a TEAM of four warps (one per SM sub-partition) owns a 16-point sub-tile: the tile E (16 k-steps x 2 point tiles,
//     8 KB, in DMMA B-fragment order) is generated cooperatively into shared memory (warp j: k-steps klo + j, + 4, ...)
//     and read back as B fragments, so no warp holds it in registers: 64 registers per thread, 32 warps per SM;
//   * the eight row blocks of a triangular operand are split {7,0} {6,1} {5,2} {4,3} over the team's warps (equal
//     dense work), the dense candidate / g rows go to the warp whose row blocks see least of the band; each warp's
//     partial |v|^2 is parked per warp and summed in warp order (deterministic);
//   * the relevance band is a contiguous k-step range [klo, khi) (the setup kernel sorts the observations), computed
//     once per super-tile from the hull of its points; loops are rolled with run-time bounds at k-step granularity (the
//     first-generation kernel skips in pairs / groups of four), so the code is small (no instruction-cache misses);
//   * phases of a team are separated by named barriers (bar.sync id, 128): eight teams per SM drift freely against each
//     other, so one team's latency-bound phases overlap the others' pipe-bound ones.
#include <cstdlib>

#include "bq_common.cuh"

namespace bqb {
namespace team {

constexpr int KS = 16;            // k-steps of the class (64 observations)
constexpr int TW = 4;             // warps per team
constexpr int ROW_Q = 0, ROW_QT = 1, ROW_TM = 2, ROW_CLOSE = 3, ROW_DENSE = 4;

__device__ __forceinline__ void team_sync(int team) {
    asm volatile("bar.sync %0, %1;" ::"r"(1 + team), "n"(TW * 32) : "memory");
}
__device__ __forceinline__ void async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ int float_key(float f) {          // order-preserving map float -> int
    const int i = __float_as_int(f);
    return i >= 0 ? i : (i ^ 0x7fffffff);
}
__device__ __forceinline__ float key_float(int k) { return __int_as_float(k >= 0 ? k : (k ^ 0x7fffffff)); }

// CTA-wide copy of `count` doubles (multiple of 2) global -> shared
__device__ __forceinline__ void stage(double *dst, const double *__restrict__ src, int count, int threads) {
    const double2 *s2 = reinterpret_cast<const double2 *>(src);
    double2 *d2 = reinterpret_cast<double2 *>(dst);
    for (int i = threadIdx.x; i < count / 2; i += threads) d2[i] = __ldg(s2 + i);
}

// Relevant k-step ranges [klo, khi) of both kernels for the points of a super-tile (same criterion as gen_masks of
// bq_score.cu: an observation can matter for some point of the hull only if (|x_s[k] - c| - hw)^2 <= reach^2 + cut, with c,
// hw the centre and half-width of the hull and reach = hw + distance from c to its nearest observation).  The
// observations are sorted, so the relevant ones are an interval.  Every lane of every warp of the team computes the same
// result.  PTS / 32 points per lane.
template <int PTS>
__device__ __forceinline__ void gen_band(const double *xrow, int npts, long long base, int na, double cut_l, double cut_tl, int nsp, int lane,
                                         const double *s_xs, int &klo_l, int &khi_l, int &klo_t, int &khi_t) {
    int klo = 0x7fffffff, khi = (int)0x80000000;
#pragma unroll
    for (int i = 0; i < PTS / 32; ++i) {
        const int p = 32 * i + lane;
        const double xv = xrow[p];
        const bool valid = p < npts && base + p < na && isfinite(xv);
        const double xc = fmin(fmax(xv, -1e30), 1e30);
        if (valid) {
            klo = min(klo, float_key(__double2float_rd(xc)));
            khi = max(khi, float_key(__double2float_ru(xc)));
        }
    }
    const double xlo = (double)key_float(__reduce_min_sync(0xffffffffu, klo));
    const double xhi = (double)key_float(__reduce_max_sync(0xffffffffu, khi));
    klo_l = khi_l = klo_t = khi_t = 0;
    if (!(xlo <= xhi)) return;                                   // no valid point
    const double c = 0.5 * (xlo + xhi), hw = 0.5 * (xhi - xlo);
    double dk[2];
    double dmin = INFINITY;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const int k = 32 * i + lane;
        dk[i] = (k < nsp) ? fabs(s_xs[k] - c) : INFINITY;        // padded observations sit at 1e150
        dmin = fmin(dmin, dk[i]);
    }
    const float dcf = __int_as_float(__reduce_min_sync(0xffffffffu, __float_as_int(__double2float_ru(fmin(dmin, 3e38)))));
    const double reach = (double)dcf + hw;
    const double r2_l = fma(reach, reach, cut_l), r2_t = fma(reach, reach, cut_tl);      // inf for cut = inf (dense)
    unsigned long long ml = 0, mt = 0;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const double t = fmax(dk[i] - hw, 0.0), t2 = t * t;
        const bool in = 32 * i + lane < nsp;
        ml |= (unsigned long long)__ballot_sync(0xffffffffu, in && t2 <= r2_l) << (32 * i);
        mt |= (unsigned long long)__ballot_sync(0xffffffffu, in && t2 <= r2_t) << (32 * i);
    }
    if (ml) { klo_l = (__ffsll((long long)ml) - 1) >> 2; khi_l = (64 - __clzll((long long)ml) + 3) >> 2; }
    if (mt) { klo_t = (__ffsll((long long)mt) - 1) >> 2; khi_t = (64 - __clzll((long long)mt) + 3) >> 2; }
}

// k-steps of row block rb that lie in the band
__device__ __forceinline__ int band_len(int rb, int klo, int khi) { return max(min(khi, 2 * rb + 2) - klo, 0); }

// One row block: c += A(rb, ks) . E(ks) over ks in [k0, k1), then q += c^2.  af: fragment (rb, 0) of the operand (lane
// included); E: the team's tile, fragment (ks, nt) at E[(ks * NT + nt) * 32 + lane].
template <int NT>
__device__ __forceinline__ void row_block(const double *af, const double *E, int k0, int k1, double (&q0)[NT], double (&q1)[NT]) {
    if (k0 >= k1) return;
    double c0[NT], c1[NT];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) c0[nt] = c1[nt] = 0.0;
    const double *pa = af + k0 * 32, *pe = E + k0 * (NT * 32);
    int n = k1 - k0;
    if (n & 1) {
        const double fa = pa[0];
        double b[NT];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) b[nt] = pe[nt * 32];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) dmma(c0[nt], c1[nt], fa, b[nt]);
        pa += 32; pe += NT * 32; --n;
    }
#pragma unroll 1
    for (; n > 0; n -= 2) {                                       // two k-steps per trip: all loads ahead of the 2 NT DMMAs
        const double fa0 = pa[0], fa1 = pa[32];
        double b0[NT], b1[NT];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) { b0[nt] = pe[nt * 32]; b1[nt] = pe[(NT + nt) * 32]; }
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) dmma(c0[nt], c1[nt], fa0, b0[nt]);
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) dmma(c0[nt], c1[nt], fa1, b1[nt]);
        pa += 64; pe += 2 * NT * 32;
    }
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
        q0[nt] = fma(c0[nt], c0[nt], q0[nt]);
        q1[nt] = fma(c1[nt], c1[nt], q1[nt]);
    }
}

// Shared memory of a launch (doubles): small arrays + resident operands, then per team: E tile, partial rows, scratch
// rows of the super-tile, two rows of query points (double buffer filled by cp.async).
struct TeamSmem {
    int n_small, n_ops, e_tile, part, scr_stride, scr, xrows, per_team;
    __host__ __device__ TeamSmem(int n_small_, int ndb, int nrow, int pts, int NT) {
        const int SUBPTS = 8 * NT;
        n_small = n_small_;
        n_ops = 2 * tri_frags(KS / 2) * 32 + ndb * KS * 32;
        e_tile = KS * NT * 32;
        part = TW * SUBPTS * 3;                   // per warp: q, tm, close of the sub-tile's points
        scr_stride = pts + 8;                     // = 8 mod 16 doubles: conflict-free 16 B fragment stores
        scr = (ROW_DENSE + nrow) * scr_stride;
        xrows = 2 * pts;
        per_team = e_tile + part + scr + xrows;
    }
    __host__ __device__ size_t doubles(int teams) const { return (size_t)n_small + n_ops + (size_t)teams * per_team; }
};

// MODE as in bq_score.cu: 0 esm / em / status; 1 + fused expected variance and per-CTA argmin partials; 2 prediction.
// SUPER: sub-tiles per super-tile of a team (8: 128 points, every warp runs the tail for 32 of them; 4: 64 points, 16 each).
template <int TEAMS, int SUPER, int NT, int TABN, int MODE>
__global__ void __launch_bounds__(TEAMS *TW * 32, 1) bq_score_team_kernel(ScoreArgs a) {
    constexpr bool EPI = MODE == 1, PRED = MODE == 2;
    constexpr int SUBPTS = 8 * NT;                // points per sub-tile
    constexpr int THREADS = TEAMS * TW * 32, WARPS = TEAMS * TW;
    constexpr int PTS = SUPER * SUBPTS;           // points per super-tile of a team
    constexpr int TAILPTS = PTS / TW;             // points per warp in the tail (32 or 16)
    extern __shared__ __align__(16) double smem[];
    __shared__ __align__(16) double s_tab[TABN];
    __shared__ int s_cta_st;
    const Layout lay = a.lay;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, team = warp >> 2, tw = warp & 3;
    const int inst = a.inst0 + blockIdx.y;
    const double *M = a.models + (size_t)inst * lay.total;
    const TeamSmem L(lay.n_small, a.ndb_max, a.nrow_res, PTS, NT);

    double *s_small = smem;
    double *s_af_l = s_small + L.n_small;
    double *s_af_t = s_af_l + tri_frags(KS / 2) * 32;
    double *s_af_d = s_af_t + tri_frags(KS / 2) * 32;
    double *tbase = s_small + L.n_small + L.n_ops + (size_t)team * L.per_team;
    double *E = tbase;
    double *part = E + L.e_tile;                  // [TW][3][SUBPTS]
    double *scr = part + L.part;                  // rows of scr_stride doubles
    double *xrows = scr + L.scr;
    const int SS = L.scr_stride;

    if (tid == 0) s_cta_st = 0;
    for (int i = tid; i < TABN; i += THREADS) s_tab[i] = a.exp_tab[(TABN == 2048 ? 0 : 2048) + i];
    for (int i = tid; i < lay.n_small; i += THREADS) s_small[i] = M[i];
    __syncthreads();
    const int nc = (int)s_small[H_NC], nsp = (int)s_small[H_NSP], ndb = (int)s_small[H_NDB];
    const int nb = nsp >> 3, nks = nsp >> 2;
    stage(s_af_l, M + lay.off_af_l_tri, tri_frags(nb) * 32, THREADS);
    stage(s_af_t, M + lay.off_af_tl_tri, tri_frags(nb) * 32, THREADS);
    stage(s_af_d, M + lay.off_af_l_dense, ndb * nks * 32, THREADS);
    __syncthreads();

    const double *s_xs = s_small + lay.off_xs, *s_tol = s_small + lay.off_tol, *s_atl = s_small + lay.off_atl;
    const double nhl = s_small[H_NHL], nhtl = s_small[H_NHTL];
    const double Cl = nhl * ExpC<TABN>::INVN, Ctl = nhtl * ExpC<TABN>::INVN;
    const int dmax_l = exp_d2max_hi(nhl), dmax_tl = exp_d2max_hi(nhtl);
    const double cut_l = a.cut_arg / fabs(nhl), cut_tl = a.cut_arg / fabs(nhtl);
    const int tol2_hi = __double2hiint(s_small[H_TOL2MAX]) + 1;
    unsigned long long n_dmma = 0;

    const double *xa = a.x_a + (size_t)(inst / a.xa_group) * a.xa_stride;
    double *o_esm = a.esm ? a.esm + (size_t)inst * a.out_stride : nullptr;
    double *o_em = a.em ? a.em + (size_t)inst * a.out_stride : nullptr;
    int *o_st = a.status ? a.status + (size_t)inst * a.out_stride : nullptr;
    const int kq = lane & 3, pq = lane >> 2;

    // Work distribution (as in bq_score.cu, with teams in place of CTAs): a UNIT is one 16-point sub-tile; super-tiles of
    // SUPER units are dealt round-robin over all teams of the grid, the remainder is split at unit granularity.
    const long long n_units = ((long long)a.na + SUBPTS - 1) / SUBPTS;
    const int G = gridDim.x * TEAMS, me = blockIdx.x * TEAMS + team;
    const int full = (int)(n_units / ((long long)G * SUPER));
    const int R = (int)(n_units - (long long)full * G * SUPER);
    const long long r_lo = (long long)full * G * SUPER + ((long long)me * R) / G;
    const int r_n = (int)(((long long)(me + 1) * R) / G - ((long long)me * R) / G);
    const int n_it = full + (r_n > 0 ? 1 : 0);
    auto tile_u = [&](int it) -> long long { return it < full ? ((long long)it * G + me) * SUPER : r_lo; };
    auto tile_n = [&](int it) { return it < full ? SUPER : r_n; };
    double best_v = INFINITY;
    long long best_i = 0x7fffffffffffffffLL;

    // the team's query points of a super-tile: warp tw fetches points [32 tw, 32 tw + 32) (those that exist)
    auto fetch = [&](double *row, int it) {
        const long long b = tile_u(it) * SUBPTS;
        const int np = tile_n(it) * SUBPTS;
        const int p = 32 * tw + lane;
        if (p < PTS) {
            if (p < np && b + p < a.na) {
                const unsigned d = (unsigned)__cvta_generic_to_shared(row + p);
                asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(xa + b + p) : "memory");
            } else {
                row[p] = 0.0;
            }
        }
    };
    int xb = 0;
    if (n_it > 0) fetch(xrows, 0);
    async_commit();

    for (int it = 0; it < n_it; ++it) {
        const int nsub = tile_n(it);
        const int npts = nsub * SUBPTS;
        const long long base = tile_u(it) * SUBPTS;
        const double *xrow = xrows + PTS * xb;
        async_wait_all();
        team_sync(team);                      // the points have landed for every warp; everyone has left the previous tail
        xb ^= 1;
        if (it + 1 < n_it) fetch(xrows + PTS * xb, it + 1);
        async_commit();

        int klo_l, khi_l, klo_t, khi_t;
        gen_band<PTS>(xrow, npts, base, a.na, cut_l, cut_tl, nsp, lane, s_xs, klo_l, khi_l, klo_t, khi_t);
        khi_l = min(khi_l, nks); khi_t = min(khi_t, nks);
        // row blocks of this warp: {nb - 1 - tw, tw}; the dense rows go to the warp whose row blocks see least of the K_l band
        const int rbA = nb - 1 - tw, rbB = tw;
        int dense_w = 0, dense_w2 = 0;       // ... split by point tile between the two least loaded warps
        {
            int best = 0x7fffffff, best2 = 0x7fffffff;
#pragma unroll
            for (int j = 0; j < TW; ++j) {
                const int ra = nb - 1 - j;
                const int w = (ra >= j ? band_len(ra, klo_l, khi_l) : 0) + (ra > j ? band_len(j, klo_l, khi_l) : 0);
                if (w < best) { best2 = best; dense_w2 = dense_w; best = w; dense_w = j; }
                else if (w < best2) { best2 = w; dense_w2 = j; }
            }
        }
        if (a.work && lane == 0) {
            const int wl = (rbA >= rbB ? band_len(rbA, klo_l, khi_l) : 0) + (rbA > rbB ? band_len(rbB, klo_l, khi_l) : 0);
            const int wt = (rbA >= rbB ? band_len(rbA, klo_t, khi_t) : 0) + (rbA > rbB ? band_len(rbB, klo_t, khi_t) : 0);
            n_dmma += (unsigned long long)nsub * NT * (wl + wt + ((tw == dense_w || tw == dense_w2) ? ndb * max(khi_l - klo_l, 0) / 2 : 0));
        }

#pragma unroll 1
        for (int sub = 0; sub < nsub; ++sub) {
            const int col0 = sub * SUBPTS;
            double x[NT];
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                const double v = xrow[col0 + nt * 8 + pq];
                x[nt] = isfinite(v) ? v : 0.0;               // invalid x_a is reported by the tail (ST_XA_BAD)
            }
            double *pw = part + tw * (3 * SUBPTS);           // this warp's partial rows: q, tm, close

            // ---- K_l: this warp's k-steps of the cross-kernel tile
#pragma unroll 1
            for (int ks = klo_l + tw; ks < khi_l; ks += TW) {
                const double xs = s_xs[4 * ks + kq];
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    const double d = x[nt] - xs;
                    E[(ks * NT + nt) * 32 + lane] = exp_kernel<TABN>(d * d, Cl, dmax_l, s_tab);
                }
            }
            // (the TL partials of the previous sub-tile are summed here, under the exp phase: see below)
            team_sync(team);                                 // B1: E(K_l) complete
            {
                double q0[NT], q1[NT];
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) q0[nt] = q1[nt] = 0.0;
                if (rbA >= rbB && rbA >= 0) row_block<NT>(s_af_l + tri_frags(rbA) * 32 + lane, E + lane, klo_l, min(khi_l, 2 * rbA + 2), q0, q1);
                if (rbA > rbB) row_block<NT>(s_af_l + tri_frags(rbB) * 32 + lane, E + lane, klo_l, min(khi_l, 2 * rbB + 2), q0, q1);
                if (tw == dense_w || tw == dense_w2) {       // dense candidate / g rows: nc + 2 rows, every k-step of the band,
                    constexpr int NH = NT / 2;               // half of the sub-tile's point tiles per warp
                    const int nt0 = (tw == dense_w) ? 0 : NH;
                    for (int db = 0; db < ndb; ++db) {
                        double c0[NH], c1[NH];
#pragma unroll
                        for (int h = 0; h < NH; ++h) c0[h] = c1[h] = 0.0;
                        const double *pa = s_af_d + (db * nks + klo_l) * 32 + lane, *pe = E + (klo_l * NT + nt0) * 32 + lane;
#pragma unroll 1
                        for (int ks = klo_l; ks < khi_l; ++ks) {
                            const double fa = pa[0];
                            double b[NH];
#pragma unroll
                            for (int h = 0; h < NH; ++h) b[h] = pe[h * 32];
#pragma unroll
                            for (int h = 0; h < NH; ++h) dmma(c0[h], c1[h], fa, b[h]);
                            pa += 32; pe += NT * 32;
                        }
                        if (db * 8 + pq < a.nrow_res) {
#pragma unroll
                            for (int h = 0; h < NH; ++h)
                                *reinterpret_cast<double2 *>(scr + (ROW_DENSE + db * 8 + pq) * SS + col0 + (nt0 + h) * 8 + 2 * kq) =
                                    make_double2(c0[h], c1[h]);
                        }
                    }
                }
                // sum the 8 row slots (lanes with equal lane & 3) and park this warp's partial
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
#pragma unroll
                    for (int o = 4; o < 32; o <<= 1) {
                        q0[nt] += __shfl_xor_sync(0xffffffffu, q0[nt], o);
                        q1[nt] += __shfl_xor_sync(0xffffffffu, q1[nt], o);
                    }
                    if (pq == 0) *reinterpret_cast<double2 *>(pw + nt * 8 + 2 * kq) = make_double2(q0[nt], q1[nt]);
                }
            }
            team_sync(team);                                 // B2: everyone is done with E(K_l); the K_l partials are parked

            // ---- K_tl: tile, gp_log_l.mean (bq.py:493) and the isclose pre-filter (bq.py:456) over this warp's k-steps
            {
                double tm[NT];
                int minhi[NT];
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) { tm[nt] = 0.0; minhi[nt] = 0x7fffffff; }
#pragma unroll 1
                for (int ks = klo_t + tw; ks < khi_t; ks += TW) {
                    const double xs = s_xs[4 * ks + kq], at = s_atl[4 * ks + kq];
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        const double d = x[nt] - xs;
                        const double d2 = d * d;
                        const double e = exp_kernel<TABN>(d2, Ctl, dmax_tl, s_tab);
                        E[(ks * NT + nt) * 32 + lane] = e;
                        minhi[nt] = min(minhi[nt], __double2hiint(d2));
                        tm[nt] = fma(at, e, tm[nt]);
                    }
                }
                // the warp in turn sums the K_l partials of this sub-tile (warp order: deterministic)
                if (tw == (sub & 3) && lane < SUBPTS) {
                    double s = 0.0;
#pragma unroll
                    for (int j = 0; j < TW; ++j) s += part[j * (3 * SUBPTS) + lane];
                    scr[ROW_Q * SS + col0 + lane] = s;
                }
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    tm[nt] += __shfl_xor_sync(0xffffffffu, tm[nt], 1);
                    tm[nt] += __shfl_xor_sync(0xffffffffu, tm[nt], 2);
                    int cl = (minhi[nt] <= tol2_hi);
                    cl |= __shfl_xor_sync(0xffffffffu, cl, 1);
                    cl |= __shfl_xor_sync(0xffffffffu, cl, 2);
                    if (kq == 0) {
                        pw[SUBPTS + nt * 8 + pq] = tm[nt];
                        pw[2 * SUBPTS + nt * 8 + pq] = cl ? 1.0 : 0.0;
                    }
                }
            }
            team_sync(team);                                 // B3: E(K_tl) complete; the K_l partial rows are free again
            {
                double q0[NT], q1[NT];
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) q0[nt] = q1[nt] = 0.0;
                if (rbA >= rbB && rbA >= 0) row_block<NT>(s_af_t + tri_frags(rbA) * 32 + lane, E + lane, klo_t, min(khi_t, 2 * rbA + 2), q0, q1);
                if (rbA > rbB) row_block<NT>(s_af_t + tri_frags(rbB) * 32 + lane, E + lane, klo_t, min(khi_t, 2 * rbB + 2), q0, q1);
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
#pragma unroll
                    for (int o = 4; o < 32; o <<= 1) {
                        q0[nt] += __shfl_xor_sync(0xffffffffu, q0[nt], o);
                        q1[nt] += __shfl_xor_sync(0xffffffffu, q1[nt], o);
                    }
                    if (pq == 0) *reinterpret_cast<double2 *>(pw + nt * 8 + 2 * kq) = make_double2(q0[nt], q1[nt]);
                }
            }
            team_sync(team);                                 // B4: everyone is done with E(K_tl); all K_tl partials are parked
            // the warp in turn sums them (it reaches the next sub-tile's B1 -- after which `part` is written again -- only
            // after this)
            if (tw == ((sub + 1) & 3) && lane < SUBPTS) {
                double s = 0.0, t = 0.0, c = 0.0;
#pragma unroll
                for (int j = 0; j < TW; ++j) {
                    s += part[j * (3 * SUBPTS) + lane];
                    t += part[j * (3 * SUBPTS) + SUBPTS + lane];
                    c += part[j * (3 * SUBPTS) + 2 * SUBPTS + lane];
                }
                if (c != 0.0) {                              // exact np.isclose(x_a, x_s, atol=1e-4) for the rare points that pass
                    const double xv = xrow[col0 + lane];
                    c = 0.0;
                    if (isfinite(xv))
                        for (int k = 0; k < nsp; ++k) if (fabs(xv - s_xs[k]) <= s_tol[k]) c = 1.0;
                }
                scr[ROW_QT * SS + col0 + lane] = s;
                scr[ROW_TM * SS + col0 + lane] = t;
                scr[ROW_CLOSE * SS + col0 + lane] = c;
            }
        }
        team_sync(team);                                     // B5: every row of the super-tile is in scratch

        // ================= tail: one lane per point; warp tw takes points [TAILPTS tw, TAILPTS (tw + 1))
        const int tp = TAILPTS * tw + lane;                  // point of the super-tile
        const long long p = base + tp;
        if (lane < TAILPTS && tp < npts && p < a.na) {
            const double xv = xrow[tp];
            const double Zm = s_small[H_ZM];
            double esm, em;
            int st = ST_OK;
            if (!isfinite(xv)) {
                esm = em = nan("");
                st = ST_XA_BAD;
            } else if (!PRED && scr[ROW_CLOSE * SS + tp] != 0.0) {
                em = Zm; esm = Zm * Zm; st = ST_SHORTCUT;         // bq.py:456-459
            } else {
                const double qs = scr[ROW_Q * SS + tp], qt = scr[ROW_QT * SS + tp], tmv = scr[ROW_TM * SS + tp];
                double *dr = scr + ROW_DENSE * SS + tp;          // dense row r at dr[r * SS]; reused for v_c
                const double c_l = s_small[H_CL], thresh = s_small[H_THRESH];
                const double *s_xc = s_small + lay.off_xc;
                unsigned mask = 0;
                for (int j = 0; j < nc; ++j) {
                    const double dc = s_xc[j] - xv;
                    if (!PRED && fabs(dc) < thresh) mask |= 1u << j;     // bq.py:470 (strict <)
                    dr[j * SS] = fma(c_l, exp_kernel<TABN>(dc * dc, Cl, dmax_l, s_tab), dr[j * SS]);   // w = k_c + W k_s
                }
                double qc = 0, vg = 0, va = 0, bg = 0, kaa;
                bool pd = true;
                if (mask == 0) {
                    const double *Lc = s_small + lay.off_lcc0, *ug = s_small + lay.off_ug0, *ua = s_small + lay.off_ua0,
                                 *rd = s_small + lay.off_rd0;
                    for (int i = 0; i < nc; ++i) {
                        double s = dr[i * SS];
                        for (int k = 0; k < i; ++k) s = fma(-Lc[i * NC_MAX + k], dr[k * SS], s);
                        s *= rd[i];
                        dr[i * SS] = s;
                        qc = fma(s, s, qc); vg = fma(s, ug[i], vg); va = fma(s, ua[i], va);
                        bg = fma(ug[i], ua[i], bg);
                    }
                    kaa = s_small[H_KAA_E];
                } else {
                    // jitter on the close candidates (bq.py:471-473): refactorise the nc x nc Schur block
                    const double *S0 = s_small + lay.off_s0, *wb = s_small + lay.off_wb, *wa = s_small + lay.off_wa;
                    const double j1 = s_small[H_J1];
                    double Lc[NC_MAX * (NC_MAX + 1) / 2], ug[NC_MAX], ua[NC_MAX];
                    for (int i = 0; i < nc && pd; ++i) {
                        for (int j = 0; j <= i; ++j) {
                            double s = S0[i * NC_MAX + j];
                            if (i == j && ((mask >> i) & 1u)) s += j1;
                            for (int k = 0; k < j; ++k) s -= Lc[i * (i + 1) / 2 + k] * Lc[j * (j + 1) / 2 + k];
                            if (i == j) {
                                if (!(s > 0.0)) { pd = false; break; }
                                Lc[i * (i + 1) / 2 + i] = sqrt(s);
                            } else {
                                Lc[i * (i + 1) / 2 + j] = s / Lc[j * (j + 1) / 2 + j];
                            }
                        }
                    }
                    if (pd) {
                        for (int i = 0; i < nc; ++i) {
                            double s = dr[i * SS], sg = wb[i], sa = wa[i];
                            for (int k = 0; k < i; ++k) {
                                const double l = Lc[i * (i + 1) / 2 + k];
                                s -= l * dr[k * SS]; sg -= l * ug[k]; sa -= l * ua[k];
                            }
                            const double d = Lc[i * (i + 1) / 2 + i];
                            s /= d; sg /= d; sa /= d;
                            dr[i * SS] = s; ug[i] = sg; ua[i] = sa;
                            qc = fma(s, s, qc); vg = fma(s, sg, vg); va = fma(s, sa, va);
                            bg = fma(sg, sa, bg);
                        }
                    }
                    kaa = s_small[H_KAA_N];
                }
                const double s_ = kaa - (qs + qc);                        // Schur pivot of the new point
                if (PRED) {
                    esm = dr[(nc + 1) * SS] + va;                         // gp_l.mean(x) = K_l(x, x_sc) alpha_l
                    em = s_small[H_KTT] - qt;                             // diag gp_log_l.cov(x)
                } else if (!pd || !(s_ > 0.0)) {
                    em = Zm; esm = Zm * Zm; st = ST_NOTPD;                // bq.py:481-490
                } else {
                    const double ba = s_small[H_BA_S] + bg;               // int_K(x_sc) . alpha_P
                    const double kg = dr[nc * SS] + vg;                   // k_a . gamma_P
                    const double ka = dr[(nc + 1) * SS] + va;             // k_a . alpha_P
                    const double diff = xv - s_small[H_MU];               // int_K at the new point (gauss_c.pyx:162)
                    const double b_a = s_small[H_CB] * exp_tab<TABN>((diff * diff) * s_small[H_NHB], s_tab);
                    const double A_a = (b_a - kg) / s_;                   // bq_c.pyx:467-469
                    const double A_sc_l = ba - A_a * ka;                  // bq_c.pyx:470
                    const double tC = s_small[H_KTT] - qt;                // gp_log_l.cov(x_a)   bq.py:496
                    const double a1 = tmv + 0.5 * tC;                     // gauss_c.pyx:87
                    const double a2 = 2.0 * tmv + 2.0 * tC;
                    if (a1 > MAX_EXPONENT) {                              // bq_c.pyx:472-475
                        esm = em = INFINITY;
                    } else {
                        const double e1 = exp_tab<TABN>(a1, s_tab);
                        em = A_sc_l + A_a * e1;                           // bq_c.pyx:477
                        if (a2 > MAX_EXPONENT) {
                            esm = INFINITY;                               // bq_c.pyx:479-483
                        } else {
                            const double e2 = exp_tab<TABN>(a2, s_tab);
                            esm = (A_sc_l * A_sc_l) + (2 * A_sc_l * A_a * e1) + ((A_a * A_a) * e2);   // bq_c.pyx:485
                        }
                    }
                    if (isnan(esm) || esm < 0) st |= ST_ESM_BAD;          // bq.py:514
                    if (isnan(em)) st |= ST_EM_BAD;                       // bq.py:518
                    if (isinf(esm)) st |= ST_ESM_INF;                     // bq.py:522
                    if (isinf(em)) st |= ST_EM_INF;                       // bq.py:524
                }
            }
            const long long po = a.perm ? a.perm[p] : p;
            if (o_esm) o_esm[po] = esm;
            if (EPI) {
                const double evv = __dsub_rn(__dadd_rn(__dmul_rn(Zm, Zm), s_small[H_ZV]), esm);   // no FMA contraction: matches the host
                a.ev[po] = evv;
                if (evv < best_v || (evv == best_v && po < best_i)) { best_v = evv; best_i = po; }
            }
            if (o_em) o_em[po] = em;
            if (o_st) o_st[po] = st;
            if (st) {
                if (a.flags) atomicOr(a.flags + inst, st);
                if (a.cta_flags) atomicOr(&s_cta_st, st);
            }
        }
    }
    if (a.work && lane == 0 && n_dmma) atomicAdd(a.work, n_dmma);
    if (a.cta_flags) {
        __syncthreads();
        if (tid == 0) a.cta_flags[blockIdx.y * gridDim.x + blockIdx.x] = s_cta_st;
    }
    if (EPI) {                                              // (min, first index) of this CTA's points
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double v2 = __shfl_xor_sync(0xffffffffu, best_v, o);
            const long long i2 = __shfl_xor_sync(0xffffffffu, best_i, o);
            if (v2 < best_v || (v2 == best_v && i2 < best_i)) { best_v = v2; best_i = i2; }
        }
        __syncthreads();                                    // the teams' shared memory is free: every warp has left the tile loop
        double *rv = s_small + L.n_small + L.n_ops;
        long long *ri = reinterpret_cast<long long *>(rv + WARPS);
        if (lane == 0) { rv[warp] = best_v; ri[warp] = best_i; }
        __syncthreads();
        if (tid == 0) {
            for (int w = 1; w < WARPS; ++w)
                if (rv[w] < best_v || (rv[w] == best_v && ri[w] < best_i)) { best_v = rv[w]; best_i = ri[w]; }
            a.part_val[blockIdx.x] = best_v;
            a.part_idx[blockIdx.x] = best_i;
        }
    }
}

constexpr size_t SMEM_LIMIT = 227 * 1024;

template <int TEAMS, int SUPER, int NT, int TABN, int MODE>
static cudaError_t launch_one(ScoreArgs a, int n_inst, int sm_count, cudaStream_t stream, int *grid_x) {
    constexpr int PTS = SUPER * 8 * NT;
    const TeamSmem L(a.lay.n_small, a.ndb_max, a.nrow_res, PTS, NT);
    const size_t bytes = sizeof(double) * L.doubles(TEAMS);
    auto kern = bq_score_team_kernel<TEAMS, SUPER, NT, TABN, MODE>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return e;
    const long long n_super = ((long long)a.na + PTS - 1) / PTS;
    long long per_inst = sm_count / n_inst;                         // persistent: one CTA per SM in total, a single wave
    const long long need = (n_super + TEAMS - 1) / TEAMS;
    if (per_inst > need) per_inst = need;
    if (per_inst < 1) per_inst = 1;
    dim3 grid((unsigned)per_inst, n_inst);
    if (grid_x) *grid_x = (int)per_inst;
    kern<<<grid, TEAMS * TW * 32, bytes, stream>>>(a);
    return cudaGetLastError();
}

template <int TEAMS, int SUPER, int NT, int TABN>
static cudaError_t launch_mode(const ScoreArgs &a, int n_inst, int sm_count, cudaStream_t stream, int *grid_x) {
    if (a.predict) return launch_one<TEAMS, SUPER, NT, TABN, 2>(a, n_inst, sm_count, stream, grid_x);
    if (a.ev) return launch_one<TEAMS, SUPER, NT, TABN, 1>(a, n_inst, sm_count, stream, grid_x);
    return launch_one<TEAMS, SUPER, NT, TABN, 0>(a, n_inst, sm_count, stream, grid_x);
}

template <int TEAMS, int SUPER, int NT, int TABN>
static bool fits(const ScoreArgs &a) {
    const TeamSmem L(a.lay.n_small, a.ndb_max, a.nrow_res, SUPER * 8 * NT, NT);
    return sizeof(double) * (L.doubles(TEAMS) + TABN) + 64 <= SMEM_LIMIT;
}

}  // namespace team

// Team kernel of the 64-observation class; cudaErrorInvalidConfiguration (nothing launched) when no configuration fits the
// launch's shared-memory needs (many candidates): the caller then uses the first-generation kernel.
cudaError_t launch_score_team_64(const ScoreArgs &a_in, int n_inst, int sm_count, cudaStream_t stream, int *grid_x) {
    using namespace team;
    ScoreArgs a = a_in;
    a.nrow_res = (a.nrow_max > 0 && a.nrow_max < 8 * a.ndb_max) ? a.nrow_max : 8 * a.ndb_max;
#define BQB_TRY(T, S, N) if (fits<T, S, N, 512>(a)) return launch_mode<T, S, N, 512>(a, n_inst, sm_count, stream, grid_x);
    // measured on C2 (ms per 10^6 points): 5 teams x 32-point sub-tiles 0.298; 8 x 16 0.333; 6 x 16 0.313; 4 x 32 0.310; 6 x 32 (64-point
    // super-tiles, half-warp tails) 0.318 -- against 0.285 of the first-generation kernel
    BQB_TRY(5, 4, 4)
#undef BQB_TRY
    return cudaErrorInvalidConfiguration;
}

}  // namespace bqb
