// Scoring kernel: expected_squared_mean / expected_mean of every query point x_a
// (replaces the per-point Python loop bq.py:399-402 -> _esm_and_em bq.py:447-527 ->
//  bq_c.expected_squared_mean_and_mean bq_c.pyx:493-535 -> _esm_and_em bq_c.pyx:425-490).
//
// The reference rebuilds and refactorises the (nsc+1)^2 bordered Gram matrix for every point.
// Here the factor of K_l(x_sc, x_sc) is fixed per model instance and every point only needs the
// border:  v = L^-1 k_a,  s = (k_aa + jitter) - v.v,  A_a = (b_a - k_a.gamma) / s, ...
// Written as  V = (c L_ss^-1) E  for a tile of points, where E[k][p] = exp(-(x_p - x_s[k])^2 / 2w^2),
// this is a lower-triangular FP64 GEMM whose B operand is *generated*, not loaded:
//
//   * one warp owns 8*NT query points and ALL rows; lane l computes exactly the B-fragment element
//     it must feed to mma.m8n8k4 (k = 4 ks + (l & 3), point = l >> 2), so the cross-kernel tile
//     lives in registers (KS*NT doubles per lane) and never touches shared memory or HBM;
//   * the A operand (c L_ss^-1, the candidate rows W, g_gamma, g_alpha; and c L_tl^-1) is stored
//     by the setup kernel in fragment order, so one conflict-free LDS.64 per lane feeds NT DMMAs.
//     For ns <= 128 it is shared-memory resident for the life of the CTA; for ns <= 256 it does
//     not fit (2 x 264 KB) and the part that is needed -- the band slab, below -- is fetched with
//     TMA bulk copies completing on mbarriers (STREAM);
//   * only v.v is needed from the triangular part: accumulators are squared and summed in
//     registers, one block of 8 rows at a time, and no n x n (or n x T) intermediate is stored;
//   * a warp works on a super-tile of 32 points (32 / (8 NT) sub-tiles); per-point partial results
//     (v_s.v_s, v_t.v_t, tm, the candidate rows) are parked in a small shared-memory scratch and the
//     candidate block (nc <= 16) plus the scalar algebra then run with one point per lane;
//   * BAND SKIPPING: E decays so fast that, per point, only a short band of observations carries
//     anything at double precision.  Per super-tile a warp derives a mask of relevant k-steps (groups of
//     four observations; gen_masks) for each of the two kernels; k-steps outside it are neither
//     exponentiated (gen_exps) nor multiplied (mask-predicated / jump-table DMMA loops), and the streamed
//     variants fetch only the rows and columns of the operands that the CTA's masks touch.  The setup kernel
//     sorts the observations, so the band is contiguous.  cut_arg = +inf makes every k-step relevant.
//   * BAND-RELATIVE TILE (classes 128 / 160 / 256, template parameter BK): the register tile holds BK = 24 k-steps from
//     the warp's band start instead of all KS (128 registers, 16 warps per SM); row-block pairs below the band run a
//     branch-free rectangular loop (rect_pairs), bands that do not fit walk windows inside the row-block loop (Wide).
//
// Grid: persistent CTAs (a multiple of the SM count); super-tiles are dealt round-robin with a
// unit-granular remainder; gridDim.y = model instances (hyper-parameter sets or independent problems).
#include <cstdlib>

#include "bq_common.cuh"

namespace bqb {


// STREAM: the triangular operands are streamed through two chunk buffers of `chunk_frags` fragments (256 B each);
// launch_score picks the largest size (<= CHUNK_FRAGS_MAX) that fits next to the resident pieces.
constexpr int CHUNK_FRAGS_MAX = 256;
#ifndef BQB_REL_GK
#define BQB_REL_GK 4          // k-steps per branch-free exp group of the band-relative kernels
#endif

// ---- mbarrier + bulk-copy (TMA) primitives of the operand stream
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "MBAR_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra MBAR_DONE;\n"
        "bra MBAR_WAIT;\n"
        "MBAR_DONE:\n"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// one thread: global -> shared bulk copy (multiple of 16 B) whose completion is counted in bytes on `bar`
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, unsigned bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

constexpr int SCR_STRIDE = 40;     // doubles per scratch row: 32 points + 8 pad (conflict-free 16 B fragment stores)
constexpr int SCR_DENSE = 4;       // first dense row

// Asynchronous fetch of the 32 query points of the super-tile starting at `base` into a scratch row: one coalesced
// 256 B read per warp, global (or page-locked host memory mapped into the device address space) -> shared with no
// register staging, issued one whole super-tile ahead of its use so that even a PCIe round trip is hidden.
__device__ __forceinline__ void fetch_points(double *row, const double *__restrict__ xa, long long base, int na, int lane) {
    if (base + lane < na) {
        const unsigned d = (unsigned)__cvta_generic_to_shared(row + lane);
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(xa + base + lane) : "memory");
    } else {
        row[lane] = 0.0;
    }
}

template <int KS, int NT, int WARPS, bool STREAM, int TABN>
struct ScoreSmem {
    static constexpr int NBC = KS / 2;
    // resident: both triangles + the dense rows; streamed: two chunk buffers + the dense rows actually used
    // nb_res: row blocks actually needed by the launch's instances (<= KS / 2): the resident operands are sized at run time
    static __host__ __device__ constexpr int operands(int ndb_max, int chunk_frags, int nb_res) {
        return STREAM ? 2 * chunk_frags * 32 + ndb_max * KS * 32 : 2 * tri_frags(nb_res) * 32 + ndb_max * 2 * nb_res * 32;
    }
    // scratch per warp: padded rows 0 qs, 1 qt, 2 tm, 3 isclose, 4.. the dense rows; then two unpadded 32-point rows
    // holding the query points of this / the next super-tile (double buffer filled by cp.async)
    // nrow: dense rows kept per warp (largest nc + 2 of the launch's instances)
    static __host__ __device__ constexpr int scr(int nrow) { return (SCR_DENSE + nrow) * SCR_STRIDE + 64; }
    static __host__ __device__ constexpr int doubles(int n_small, int ndb_max, int chunk_frags, int nb_res, int nrow) {
        return n_small + operands(ndb_max, chunk_frags, nb_res) + WARPS * scr(nrow);     // dynamic part; the exp table is static
    }
};

// CTA-wide copy of `count` doubles (multiple of 2) global -> shared, 16 B per thread per step
template <int THREADS>
__device__ __forceinline__ void stage(double *dst, const double *__restrict__ src, int count) {
    const double2 *s2 = reinterpret_cast<const double2 *>(src);
    double2 *d2 = reinterpret_cast<double2 *>(dst);
    for (int i = threadIdx.x; i < count / 2; i += THREADS) d2[i] = __ldg(s2 + i);
}

// Mask of the k-steps (4 observations each) of a sub-tile that are numerically relevant: bit ks.
template <int KS> struct KMask { using type = unsigned; };
template <> struct KMask<40> { using type = unsigned long long; };
template <> struct KMask<64> { using type = unsigned long long; };

// A cross-kernel element whose exponent lies more than CUT_ARG below the largest one of its own point is below
// e^-72 = 5e-32 of that point's leading element: with cond(K) < 1e9 it cannot change any of the point's results at
// double precision (DESIGN.md, "band skipping").  K-steps in which every element of the sub-tile is that small are
// neither exponentiated nor multiplied.
constexpr double CUT_ARG = 72.0;      // the default of ScoreArgs::cut_arg (bq_common.cuh) and bqb_batch_set_cutoff
static_assert(CUT_ARG == 72.0, "keep in step with ScoreArgs::cut_arg and include/bq_b200.h");

// Cross-kernel B fragments of one sub-tile, bf[ks][nt] = exp(-(x - x_s[k])^2 / (2 w^2)), k = 4 ks + (lane & 3), are
// produced in two steps.
//
// gen_masks (once per super-tile of 32 points per warp, serves both kernels and all sub-tiles): which k-steps are
// relevant.  The per-point criterion (exponent within CUT_ARG of the point's own largest) is bounded from the hull of
// the warp's points instead of being evaluated per element: with c and hw the centre and half-width of the hull and dc
// the distance from c to its nearest observation, every point has an observation within reach = dc + hw, so an
// observation can only be relevant for some point if (|x_s[k] - c| - hw)^2 <= reach^2 + cut.  That is one comparison
// per observation (lane <-> observation, nsp / 32 steps, distances kept in registers) and a ballot per 32
// observations; the hull and dc are warp-reduced with REDUX on float-rounded values (rounded outwards: the criterion
// only has to be conservative).  The first version computed every squared distance of every sub-tile and built the
// masks bit by bit, which cost more instructions than the exponentials it saved.  For sorted query vectors (grids) the
// hull criterion selects the same k-steps as the per-point one; for scattered points it selects more (never fewer).
__device__ __forceinline__ int float_key(float f) {          // order-preserving map float -> int
    const int i = __float_as_int(f);
    return i >= 0 ? i : (i ^ 0x7fffffff);
}
__device__ __forceinline__ float key_float(int k) { return __int_as_float(k >= 0 ? k : (k ^ 0x7fffffff)); }

template <int KS>
__device__ __forceinline__ void gen_masks(double xv, bool valid, double cut_l, double cut_tl, int nsp, int lane,
                                          const double *s_xs, typename KMask<KS>::type &mask_l, typename KMask<KS>::type &mask_tl) {
    using mask_t = typename KMask<KS>::type;
    constexpr int NW = (KS + 7) / 8;                 // 32-observation words
    // hull of the warp's points (one per lane; lanes past the end or with invalid x do not count)
    const double xc = fmin(fmax(xv, -1e30), 1e30);
    const int klo = valid ? float_key(__double2float_rd(xc)) : 0x7fffffff;
    const int khi = valid ? float_key(__double2float_ru(xc)) : (int)0x80000000;
    const double xlo = (double)key_float(__reduce_min_sync(0xffffffffu, klo));
    const double xhi = (double)key_float(__reduce_max_sync(0xffffffffu, khi));
    if (!(xlo <= xhi)) { mask_l = 0; mask_tl = 0; return; }      // no valid point in this warp's tile
    const double c = 0.5 * (xlo + xhi), hw = 0.5 * (xhi - xlo);
    double dk[NW];
    double dmin = INFINITY;
#pragma unroll
    for (int i = 0; i < NW; ++i) {
        const int k = 32 * i + lane;
        dk[i] = (k < nsp) ? fabs(s_xs[k] - c) : INFINITY;        // padded observations sit at 1e150
        dmin = fmin(dmin, dk[i]);
    }
    // nearest observation to c, rounded up (positive floats order like their bits)
    const float dcf = __int_as_float(__reduce_min_sync(0xffffffffu, __float_as_int(__double2float_ru(fmin(dmin, 3e38)))));
    const double reach = (double)dcf + hw;
    const double r2_l = fma(reach, reach, cut_l), r2_tl = fma(reach, reach, cut_tl);        // inf for cut = inf (dense)
    mask_t ml = 0, mt = 0;
#pragma unroll
    for (int i = 0; i < NW; ++i) {
        const double t = fmax(dk[i] - hw, 0.0), t2 = t * t;
        const bool in = 32 * i + lane < nsp;
        unsigned bl = __ballot_sync(0xffffffffu, in && t2 <= r2_l), bt = __ballot_sync(0xffffffffu, in && t2 <= r2_tl);
        // observation bits -> k-step bits: k-step j of this word is relevant if any of bits 4j .. 4j+3 is set
        bl |= bl >> 1; bl |= bl >> 2; bl &= 0x11111111u;
        bl = (bl | (bl >> 3)) & 0x03030303u; bl = (bl | (bl >> 6)) & 0x000f000fu; bl = (bl | (bl >> 12)) & 0xffu;
        bt |= bt >> 1; bt |= bt >> 2; bt &= 0x11111111u;
        bt = (bt | (bt >> 3)) & 0x03030303u; bt = (bt | (bt >> 6)) & 0x000f000fu; bt = (bt | (bt >> 12)) & 0xffu;
        ml |= (mask_t)bl << (8 * i);
        mt |= (mask_t)bt << (8 * i);
    }
    mask_l = ml;
    mask_tl = mt;
}

// gen_exps computes the squared distances and exponentials of the relevant k-steps (9 FP64 + 6 integer instructions per
// element): groups of GK k-steps are branch free so that GK NT independent exp chains interleave, and a group runs if
// any of its k-steps is relevant.  The K_tl pass also accumulates gp_log_l.mean (bq.py:493) and pre-filters
// np.isclose(x_a, x_s, atol=1e-4) (bq.py:456): the high word of the point's smallest d^2 (its nearest observation is
// always in a relevant k-step) against an upper bound of every tolerance^2 -- non-negative doubles order like their
// bits; the exact test runs afterwards only for the rare points that pass (isclose_exact).
template <int NT> __host__ __device__ constexpr int exp_group() { return NT == 1 ? 8 : 4; }
template <int KS, int NT, int TABN, bool TL, int GK = exp_group<NT>()>
__device__ __forceinline__ void gen_exps(double (&bf)[KS][NT], const double (&x)[NT], double C, int d2max_hi,
                                         typename KMask<KS>::type mask, int kq, const double *s_xs, const double *s_atl,
                                         const double *s_tab, double (&tm)[NT], int tol2_hi, int (&close)[NT], int nkv = KS) {
    using mask_t = typename KMask<KS>::type;
    // 8 independent exp chains per branch-free group: with one CTA of 8 warps per SM (two warps per scheduler) the
    // NT = 1 exp phase was latency bound at 4 (ncu: 47 % of its stalls on fixed-latency dependencies)
    int minhi[NT];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) minhi[nt] = 0x7fffffff;
#pragma unroll
    for (int g = 0; g < (KS + GK - 1) / GK; ++g) {
        if ((mask >> (GK * g)) & (((mask_t)1 << GK) - 1)) {
#pragma unroll
            for (int j = 0; j < GK; ++j) {
                const int ks = GK * g + j;
                if (ks < KS) {
                    const double xs = s_xs[4 * ks + kq];
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        const double d = x[nt] - xs;
                        const double d2 = d * d;
                        const double e = exp_kernel<TABN>(d2, C, d2max_hi, s_tab);
                        bf[ks][nt] = e;
                        if (TL) {
                            minhi[nt] = min(minhi[nt], __double2hiint(d2));
                            // nkv: k-steps of the tile that exist (a band-relative tile may reach past the class capacity:
                            // such elements are generated from padding and never multiplied, but must not enter the mean)
                            if (ks < nkv) tm[nt] = fma(s_atl[4 * ks + kq], e, tm[nt]);
                        }
                    }
                }
            }
        }
    }
    if (TL) {
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) close[nt] = (minhi[nt] <= tol2_hi);      // per lane; the caller ORs the four k residues
    }
}

// Exact np.isclose(x_a, x_s, atol=1e-4): |x_a - x_s[k]| <= 1e-4 + 1e-5 |x_s[k]| for this lane's k residues (padded
// entries carry tolerance -1).  Rolled loop: it only runs for points that passed the pre-filter.
__device__ __forceinline__ int isclose_exact(double x, const double *s_xs, const double *s_tol, int nsp, int kq) {
    int c = 0;
    for (int k = kq; k < nsp; k += 4) c |= (fabs(x - s_xs[k]) <= s_tol[k]);
    return c;
}

// cp.async group bookkeeping of the query-point prefetch (fetch_points)
__device__ __forceinline__ void async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// One block of 8 rows: acc = A(rb, 0 .. lim-1) . B, then q += acc^2.  The k-step loop is unrolled at compile
// time (B fragments are registers) and leaves early at the row block's diagonal, so the row-block loop
// around it can stay rolled: the instruction footprint is KS DMMAs, not KS^2/2.
template <int KS, int NT>
__device__ __forceinline__ void row_block_acc(const double *af, int lim, const double (&bf)[KS][NT], double (&c0)[NT],
                                              double (&c1)[NT], double (&e0)[NT], double (&e1)[NT],
                                              typename KMask<KS>::type mask) {
    using mask_t = typename KMask<KS>::type;
    constexpr bool DUAL = (NT == 1);    // NT == 1: split even / odd k-steps into two chains to cover the DMMA latency
#pragma unroll
    for (int ks = 0; ks < KS; ks += 2) {
        if (ks >= lim) break;
        if (mask & ((mask_t)3 << ks)) {              // warp-uniform: a relevant k-step in this pair
            const double a0 = af[ks * 32], a1 = af[(ks + 1) * 32];
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                dmma(c0[nt], c1[nt], a0, bf[ks][nt]);
                if (DUAL) dmma(e0[nt], e1[nt], a1, bf[ks + 1][nt]);
                else dmma(c0[nt], c1[nt], a1, bf[ks + 1][nt]);
            }
        }
    }
}
template <int NT>
__device__ __forceinline__ void row_block_finish(const double (&c0)[NT], const double (&c1)[NT], const double (&e0)[NT],
                                                 const double (&e1)[NT], double (&q0)[NT], double (&q1)[NT]) {
    constexpr bool DUAL = (NT == 1);
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
        const double r0 = DUAL ? c0[nt] + e0[nt] : c0[nt], r1 = DUAL ? c1[nt] + e1[nt] : c1[nt];
        q0[nt] = fma(r0, r0, q0[nt]);
        q1[nt] = fma(r1, r1, q1[nt]);
    }
}
template <int KS, int NT>
__device__ __forceinline__ void row_block(const double *af, int lim, const double (&bf)[KS][NT], double (&q0)[NT],
                                          double (&q1)[NT], typename KMask<KS>::type mask) {
    double c0[NT], c1[NT], e0[NT], e1[NT];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) { c0[nt] = c1[nt] = e0[nt] = e1[nt] = 0.0; }
    row_block_acc<KS, NT>(af, lim, bf, c0, c1, e0, e1, mask);
    row_block_finish<NT>(c0, c1, e0, e1, q0, q1);
}

// Two consecutive row blocks at once (rolled loops): the B fragment of a k-step feeds both, which doubles the number
// of independent DMMA chains per warp, and the k loop advances four k-steps per (branch-free) group so that the eight
// A-fragment loads of a group are issued ahead of its DMMAs.  ncu on the ns = 256 kernel had 42 % of the DMMA-phase
// stalls on the LDS -> DMMA scoreboard and one ISETP + BRA per two DMMAs with the one-block-at-a-time loop.
// limA = k-steps of the first row block (2 rb + 2); the second one has two more.
//
// pair_group is the group of four k-steps starting at the compile-time k-step K0 (the B fragments are registers).
template <int KS, int NT, int K0>
__device__ __forceinline__ void pair_group(const double *afA, const double *afB, int limA, const double (&bf)[KS][NT],
                                           double (&a0)[NT], double (&a1)[NT], double (&b0)[NT], double (&b1)[NT],
                                           double (&c0)[NT], double (&c1)[NT], double (&d0)[NT], double (&d1)[NT]) {
    constexpr int ks = K0;
    if (ks + 4 <= limA) {
        double fa[4], fb[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) { fa[j] = afA[(ks + j) * 32]; fb[j] = afB[(ks + j) * 32]; }
#pragma unroll
        for (int j = 0; j < 4; j += 2)
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                dmma(a0[nt], a1[nt], fa[j], bf[ks + j][nt]);
                dmma(c0[nt], c1[nt], fb[j], bf[ks + j][nt]);
                dmma(b0[nt], b1[nt], fa[j + 1], bf[ks + j + 1][nt]);
                dmma(d0[nt], d1[nt], fb[j + 1], bf[ks + j + 1][nt]);
            }
    } else if (ks + 2 <= limA) {             // limA == ks + 2: two more k-steps for both, then B's last two
        const double fa0 = afA[ks * 32], fa1 = afA[(ks + 1) * 32];
        double fb[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) fb[j] = afB[(ks + j) * 32];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            dmma(a0[nt], a1[nt], fa0, bf[ks][nt]);
            dmma(c0[nt], c1[nt], fb[0], bf[ks][nt]);
            dmma(b0[nt], b1[nt], fa1, bf[ks + 1][nt]);
            dmma(d0[nt], d1[nt], fb[1], bf[ks + 1][nt]);
            dmma(c0[nt], c1[nt], fb[2], bf[ks + 2][nt]);
            dmma(d0[nt], d1[nt], fb[3], bf[ks + 3][nt]);
        }
    } else {                                 // limA == ks: only B's last two k-steps remain
        const double fb0 = afB[ks * 32], fb1 = afB[(ks + 1) * 32];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            dmma(c0[nt], c1[nt], fb0, bf[ks][nt]);
            dmma(d0[nt], d1[nt], fb1, bf[ks + 1][nt]);
        }
    }
}

// [g0, kend): first relevant group of four k-steps and the end (a multiple of 4) of the last one, from the mask.  The
// groups are entered through a jump table at g0 and left at kend or at the diagonal: with a band of 2-4 groups out of up
// to 16, testing every group of every row-block pair cost more than the DMMAs (ncu, ns = 256).
// PLAIN: the band is groups 0 .. kend / 4 - 1 without holes (plain_band): straight-line code from group 0, no jump table.
template <int KS, int NT, bool PLAIN = false>
__device__ __forceinline__ void row_block_pair(const double *afA, const double *afB, int limA, const double (&bf)[KS][NT],
                                               double (&q0)[NT], double (&q1)[NT], typename KMask<KS>::type mask, int g0, int kend) {
    using mask_t = typename KMask<KS>::type;
    static_assert(KS % 4 == 0 && KS <= 64, "k-steps come in groups of 4, at most 16 groups");
    double a0[NT], a1[NT], b0[NT], b1[NT], c0[NT], c1[NT], d0[NT], d1[NT];   // (a, b): block A even / odd k; (c, d): block B
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) { a0[nt] = a1[nt] = b0[nt] = b1[nt] = c0[nt] = c1[nt] = d0[nt] = d1[nt] = 0.0; }
    const int kstop = min(kend, limA + 2);   // both row blocks are complete at limA + 2
#define BQB_GRP(G)                                                                                                       \
    case G:                                                                                                              \
        if constexpr (4 * (G) < KS) {                                                                                    \
            if (4 * (G) >= kstop) break;                                                                                 \
            if (mask & ((mask_t)15 << (4 * (G))))      /* holes: observations need not be sorted */                      \
                pair_group<KS, NT, 4 * (G)>(afA, afB, limA, bf, a0, a1, b0, b1, c0, c1, d0, d1);                         \
        }                                                                                                                \
        [[fallthrough]];
#define BQB_GRP_PLAIN(G)                                                                                                 \
    if constexpr (4 * (G) < KS) {                                                                                        \
        if (4 * (G) < kstop) {                                                                                           \
            pair_group<KS, NT, 4 * (G)>(afA, afB, limA, bf, a0, a1, b0, b1, c0, c1, d0, d1);
    if constexpr (PLAIN) {      // nested: group G + 1 only if group G ran
        BQB_GRP_PLAIN(0) BQB_GRP_PLAIN(1) BQB_GRP_PLAIN(2) BQB_GRP_PLAIN(3) BQB_GRP_PLAIN(4) BQB_GRP_PLAIN(5) BQB_GRP_PLAIN(6) BQB_GRP_PLAIN(7)
        }} }} }} }} }} }} }} }}
    } else {
        switch (g0) {
            BQB_GRP(0) BQB_GRP(1) BQB_GRP(2) BQB_GRP(3) BQB_GRP(4) BQB_GRP(5) BQB_GRP(6) BQB_GRP(7)
            BQB_GRP(8) BQB_GRP(9) BQB_GRP(10) BQB_GRP(11) BQB_GRP(12) BQB_GRP(13) BQB_GRP(14) BQB_GRP(15)
            default: break;
        }
    }
#undef BQB_GRP_PLAIN
#undef BQB_GRP
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
        const double rA0 = a0[nt] + b0[nt], rA1 = a1[nt] + b1[nt], rB0 = c0[nt] + d0[nt], rB1 = c1[nt] + d1[nt];
        q0[nt] = fma(rA0, rA0, q0[nt]);
        q1[nt] = fma(rA1, rA1, q1[nt]);
        q0[nt] = fma(rB0, rB0, q0[nt]);
        q1[nt] = fma(rB1, rB1, q1[nt]);
    }
}

// first relevant group of four k-steps / end of the last one
template <typename mask_t>
__device__ __forceinline__ void mask_groups(mask_t mask, int &g0, int &kend) {
    const unsigned long long m = mask;
    g0 = (__ffsll((long long)m) - 1) >> 2;
    kend = (64 - __clzll((long long)m) + 3) & ~3;
}

// The rectangular part of a band-relative pass: row-block pairs that lie wholly below the band see all of it, here as NP
// pairs of k-steps (bf[0 .. 2 NP)), so the loop needs no diagonal tests, no jump table and no per-pair address
// arithmetic: per row-block pair 4 NP fragment loads, 4 NP NT DMMAs in four independent chains per point tile (the first
// DMMA of a chain starts from a zero accumulator), four adds and four FMAs.  ncu on the generic loop (ns = 256): 14.5
// instructions per DMMA, among them ~40 of address arithmetic and 17 accumulator clears per pair; this loop issues ~3.5.
// pA: fragment (rb, k0) of the pair's first row block (lane included); the second row block starts sAB doubles later, the
// next pair sNext doubles later, and both distances grow by dAB / dNext per pair (resident triangles: rows get longer;
// slabs: constant row pitch).
__device__ __forceinline__ void dmma_z(double &c0, double &c1, double a, double b) {      // D = A B (zero accumulator)
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%4,%5};"
                 : "=d"(c0), "=d"(c1) : "d"(a), "d"(b), "d"(0.0), "d"(0.0));
}
template <int KS, int NT, int NP>        // NP: pairs of k-steps (bf[0 .. 2 NP))
__device__ __forceinline__ void rect_pairs(const double *pA, int npair, int sAB, int sNext, int dAB, int dNext,
                                           const double (&bf)[KS][NT], double (&q0)[NT], double (&q1)[NT]) {
    static_assert(2 * NP <= KS, "k-step pairs of the register tile");
#pragma unroll 1
    for (int i = 0; i < npair; ++i) {
        const double *pB = pA + sAB;
        double a0[NT], a1[NT], b0[NT], b1[NT], c0[NT], c1[NT], d0[NT], d1[NT];   // (a, b): block A even / odd k; (c, d): block B
#pragma unroll
        for (int u = 0; u < NP; ++u) {
            const double fa0 = pA[(2 * u) * 32], fa1 = pA[(2 * u + 1) * 32], fb0 = pB[(2 * u) * 32], fb1 = pB[(2 * u + 1) * 32];
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                if (u == 0) {
                    dmma_z(a0[nt], a1[nt], fa0, bf[0][nt]);
                    dmma_z(c0[nt], c1[nt], fb0, bf[0][nt]);
                    dmma_z(b0[nt], b1[nt], fa1, bf[1][nt]);
                    dmma_z(d0[nt], d1[nt], fb1, bf[1][nt]);
                } else {
                    dmma(a0[nt], a1[nt], fa0, bf[2 * u][nt]);
                    dmma(c0[nt], c1[nt], fb0, bf[2 * u][nt]);
                    dmma(b0[nt], b1[nt], fa1, bf[2 * u + 1][nt]);
                    dmma(d0[nt], d1[nt], fb1, bf[2 * u + 1][nt]);
                }
            }
        }
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            const double rA0 = a0[nt] + b0[nt], rA1 = a1[nt] + b1[nt], rB0 = c0[nt] + d0[nt], rB1 = c1[nt] + d1[nt];
            q0[nt] = fma(rA0, rA0, q0[nt]);
            q1[nt] = fma(rA1, rA1, q1[nt]);
            q0[nt] = fma(rB0, rB0, q0[nt]);
            q1[nt] = fma(rB1, rB1, q1[nt]);
        }
        pA += sNext;
        sAB += dAB;
        sNext += dNext;
    }
}
template <int KS, int NT>
__device__ __forceinline__ void rect_dispatch(int np, const double *pA, int npair, int sAB, int sNext, int dAB, int dNext,
                                              const double (&bf)[KS][NT], double (&q0)[NT], double (&q1)[NT]) {
    switch (np) {
#define BQB_RECT(N)                                                                                          \
    case N:                                                                                                  \
        if constexpr (2 * (N) <= KS) rect_pairs<KS, NT, (2 * (N) <= KS ? (N) : 1)>(pA, npair, sAB, sNext, dAB, dNext, bf, q0, q1); \
        break;
        BQB_RECT(1) BQB_RECT(2) BQB_RECT(3) BQB_RECT(4) BQB_RECT(5) BQB_RECT(6) BQB_RECT(7) BQB_RECT(8)
        BQB_RECT(9) BQB_RECT(10) BQB_RECT(11) BQB_RECT(12) BQB_RECT(13) BQB_RECT(14) BQB_RECT(15) BQB_RECT(16)
#undef BQB_RECT
        default: break;
    }
}
// The band of a relative mask is "plain" when its groups of four k-steps are 0 .. ng-1 without holes: every bf of
// those groups has been generated, so the rectangular loop may multiply them all.
template <typename mask_t>
__device__ __forceinline__ bool plain_band(mask_t mask, int g0, int kend) {
    unsigned long long m = mask;
    m |= m >> 1; m |= m >> 2; m &= 0x1111111111111111ull;            // bit 4 g: group g relevant
    const unsigned long long want = (kend >= 64 ? ~0ull : ((1ull << kend) - 1)) & 0x1111111111111111ull;
    return g0 == 0 && m == want;
}

// ---- BAND-RELATIVE register tile (template parameter BK > 0 of the kernel).  The cross-kernel tile of a sub-tile holds
// only KB = BK k-steps starting at the warp's band start k0 (a multiple of 8 k-steps, from the relevance mask of the
// warp's 32 points): bf[j] is k-step k0 + j, the relevance mask is shifted down by k0 and the A-fragment pointers are
// advanced by k0 fragments, so every loop below runs unchanged on relative indices.  The register tile no longer grows
// with the capacity class (KB NT doubles instead of KS NT), which is what lets 16 warps share an SM.
//
// A warp whose band does not fit (scattered query points, length scales of many observation spacings, cut_arg = inf)
// takes the WIDE path: the band is walked in windows of KB k-steps *inside* the row-block loop, the window's exponentials
// being regenerated for every row block (accumulators must see the whole band before they are squared).  Slow -- the
// exponentials are recomputed n / 8 times -- but it keeps every launch correct for any input without a second kernel.
template <int NT>
struct Wide {
    bool on;                      // this warp's band exceeds the register tile in this pass
    unsigned long long mask;      // absolute relevance mask of the warp
    int kbeg, kend;               // band [kbeg, kend) in k-steps, kbeg a multiple of 8
    double x[NT];
    double C;
    int dmax, kq;
    const double *s_xs, *s_tab;
};
// window [kw, kw + KB) of the absolute mask, as a relative mask
template <int KB>
__device__ __forceinline__ typename KMask<KB>::type window_mask(unsigned long long mask, int kw) {
    const unsigned long long m = mask >> kw;
    return (typename KMask<KB>::type)(KB >= 64 ? m : (m & ((1ull << (KB & 63)) - 1)));
}
// one row block on the wide path; af[ks * 32] = fragment (rb, ks) with ABSOLUTE ks, lim = 2 rb + 2
template <int KB, int NT, int TABN>
__device__ __forceinline__ void wide_row_block(const double *af, int lim, const Wide<NT> &w, double (&bf)[KB][NT],
                                               double (&q0)[NT], double (&q1)[NT]) {
    double c0[NT], c1[NT], e0[NT], e1[NT], tmd[NT];
    int cld[NT];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) { c0[nt] = c1[nt] = e0[nt] = e1[nt] = 0.0; }
    const int kstop = min(w.kend, lim);
#pragma unroll 1
    for (int kw = w.kbeg; kw < kstop; kw += KB) {
        const typename KMask<KB>::type rm = window_mask<KB>(w.mask, kw);
        if (!rm) continue;
        gen_exps<KB, NT, TABN, false>(bf, w.x, w.C, w.dmax, rm, w.kq, w.s_xs + 4 * kw, nullptr, w.s_tab, tmd, 0, cld);
        row_block_acc<KB, NT>(af + kw * 32, lim - kw, bf, c0, c1, e0, e1, rm);
    }
    row_block_finish<NT>(c0, c1, e0, e1, q0, q1);
}

// Row blocks [rb0, rb1) of a triangular operand whose fragment (rb, ks) sits at base[(tri_frags(rb) + ks) * 32].
// KS is the size of the register tile bf, k0 its first k-step (0 for the absolute tile) and `mask` is relative to k0.
template <int KS, int NT, int TABN, bool REL>
__device__ __forceinline__ void row_blocks_rolled(const double *base, int rb0, int rb1, double (&bf)[KS][NT],
                                                  double (&q0)[NT], double (&q1)[NT], typename KMask<KS>::type mask, int k0,
                                                  const Wide<NT> &w) {
    if constexpr (REL) {
        if (w.on) {
            const int kfirst = __ffsll((long long)w.mask) - 1;
#pragma unroll 1
            for (int rb = max(rb0, kfirst >> 1); rb < rb1; ++rb)
                wide_row_block<KS, NT, TABN>(base + tri_frags(rb) * 32, 2 * rb + 2, w, bf, q0, q1);
            return;
        }
    }
    if (!mask) return;
    int g0, kend;
    mask_groups(mask, g0, kend);
    const int kfirst = k0 + __ffsll((long long)(unsigned long long)mask) - 1;      // first relevant k-step (absolute)
    int rb = rb0;
    // REL: pairs from rbf on lie below the band (2 rb + 2 - k0 >= kend) and take the rectangular loop
    const bool rect = REL && plain_band(mask, g0, kend);
    const int kend2 = (64 - __clzll((long long)(unsigned long long)mask) + 1) & ~1;      // band end rounded to a pair of k-steps
    const int rbf = rect ? min(rb1, max(rb0, ((k0 + kend2) >> 1) & ~1)) : rb1;
#pragma unroll 1
    for (; rb + 1 < rbf; rb += 2) {
        // rows above the first relevant k-step see none of it (lower-triangular operand): 2 rb + 4 k-steps at most
        if (2 * rb + 4 <= kfirst) continue;
        if (REL && rect)
            row_block_pair<KS, NT, REL>(base + (tri_frags(rb) + k0) * 32, base + (tri_frags(rb + 1) + k0) * 32, 2 * rb + 2 - k0, bf, q0, q1,
                                        mask, g0, kend);
        else
            row_block_pair<KS, NT>(base + (tri_frags(rb) + k0) * 32, base + (tri_frags(rb + 1) + k0) * 32, 2 * rb + 2 - k0, bf, q0, q1,
                                   mask, g0, kend);
    }
    if constexpr (REL) {
        if (rect && rb + 1 < rb1) {
            const int npair = (rb1 - rb) >> 1;
            rect_dispatch<KS, NT>(kend2 >> 1, base + (tri_frags(rb) + k0) * 32, npair, (2 * rb + 2) * 32, (4 * rb + 6) * 32, 128, 256, bf,
                                  q0, q1);
            rb += 2 * npair;
        }
    }
    if (rb < rb1) row_block<KS, NT>(base + (tri_frags(rb) + k0) * 32, 2 * rb + 2 - k0, bf, q0, q1, mask);
}

// (row block, k-step) products a triangular pass executes for a relevance mask: sum over row blocks rb < nb of
// popc(mask & low(2 rb + 2)), at the pair granularity of the DMMA loops.  Only used for the work counter.
template <int KS>
__device__ __forceinline__ unsigned count_ksteps(typename KMask<KS>::type mask, int nb) {
    unsigned long long m = mask;
    m = (m | (m >> 1)) & 0x5555555555555555ull;              // a pair runs if either k-step is relevant ...
    m |= m << 1;                                             // ... and then both are multiplied
    unsigned n = 0;
    for (int rb = 0; rb < nb; ++rb) n += __popcll(2 * rb + 2 >= 64 ? m : (m & ((1ull << (2 * rb + 2)) - 1)));
    return n;
}

// Lower-triangular pass with shared-memory resident operands: q += (rows of (A . B))^2.
// ROLLED = false unrolls the row-block loop as well (exact trip counts, no early-exit branches).
// Phase alignment of the ns <= 64 kernels: the warps of a barrier group enter the exp and the DMMA phases together
// (DMMA / DFMA mixing on an SMSP costs pipe throughput).  ALIGN = 0: free running; 1: the whole CTA (__syncthreads);
// N >= 2: groups of N consecutive warps on their own named barrier, so that the groups of a CTA drift apart and one
// group's latency-bound phases (relevance masks, per-point tail) overlap the other groups' pipe-bound ones.
template <int ALIGN>
__device__ __forceinline__ void phase_sync() {
    if constexpr (ALIGN == 1) __syncthreads();
    else if constexpr (ALIGN > 1)
        asm volatile("bar.sync %0, %1;" ::"r"(1 + (int)(threadIdx.x >> 5) / ALIGN), "n"(ALIGN * 32) : "memory");
}

template <int KS, int NT, int TABN, int ALIGN, bool ROLLED, bool REL>
__device__ __forceinline__ void tri_pass(const double *af_res, double (&bf)[KS][NT], double (&q0)[NT], double (&q1)[NT],
                                         int nb, int lane, typename KMask<KS>::type mask, int k0, const Wide<NT> &w) {
    using mask_t = typename KMask<KS>::type;
    static_assert(ROLLED || !REL, "the band-relative tile needs the rolled row-block loop");
    phase_sync<ALIGN>();                                        // the warps of a barrier group enter the DMMA phase together
    if constexpr (ROLLED) {
        row_blocks_rolled<KS, NT, TABN, REL>(af_res + lane, 0, nb, bf, q0, q1, mask, k0, w);
    } else {
#pragma unroll
        for (int rb = 0; rb < KS / 2; ++rb) {      // lim is a compile-time constant after unrolling: the early exit folds away
            constexpr int BITS = 8 * sizeof(mask_t);
            const mask_t low = (2 * rb + 2 >= BITS) ? ~(mask_t)0 : (((mask_t)1 << (2 * rb + 2)) - 1);
            if (rb < nb && (mask & low)) row_block<KS, NT>(af_res + tri_frags(rb) * 32 + lane, 2 * rb + 2, bf, q0, q1, mask);
        }
    }
}

// Streamed variant (operands do not fit in shared memory).  Only the *band slab* of a triangular operand is needed for
// a sub-tile: the row blocks rb >= klo / 2 and, of each, the k-steps [klo, khi) that are relevant for any warp of the
// CTA (klo aligned to the 4-k-step groups of the DMMA loops).  A slab chunk is up to R such row blocks, each one bulk
// copy (TMA) of W = khi - klo fragments issued by one lane of warp 0 and completing, in bytes, on the buffer's mbarrier;
// two chunk buffers alternate, so that the next chunk (of this operand or of the next one) lands while the CTA's warps
// run the DMMAs of the current one.  A row block that reaches its diagonal before khi copies a few fragments of the
// next row block (same array, unused).  With every k-step relevant this degenerates to streaming whole rows.
// (History: per-thread cp.async staging cost ~16 LDGSTS + address arithmetic per thread and chunk, each LDGSTS batch
// preceded by three dummy LDS in the SASS, and two CTA barriers per chunk; whole-operand TMA chunks were latency
// bound once band skipping had removed most of the arithmetic.)
struct SlabPlan {
    int klo, W, rb_first, R, nchunk;
};
template <int KS>
__device__ __forceinline__ SlabPlan make_slab_plan(typename KMask<KS>::type um, int nks, int nb, int cap_frags) {
    SlabPlan p;
    if (um == 0) { p.klo = p.W = p.rb_first = p.R = p.nchunk = 0; return p; }
    const unsigned long long m = um;
    const int lo = __ffsll((long long)m) - 1, hi = 64 - __clzll((long long)m);      // relevant k-steps lie in [lo, hi)
    p.klo = lo & ~3;
    const int khi = min((hi + 3) & ~3, nks);
    p.W = khi - p.klo;
    p.rb_first = p.klo >> 1;                          // even: row blocks are consumed in pairs
    p.R = max(2, (cap_frags / p.W) & ~1);
    p.nchunk = (nb - p.rb_first + p.R - 1) / p.R;
    return p;
}
struct Stream {
    unsigned long long *bar;      // [2] "chunk landed" barriers, one per buffer
    double *buf;                  // two buffers of `stride` doubles
    int stride;
    unsigned phase;               // bit b: parity to wait for on buffer b
};
// warp 0, all lanes: issue slab chunk c of `op` into buffer `b`
__device__ __forceinline__ void slab_issue(const double *__restrict__ op, const SlabPlan &p, int c, int nb, const Stream &st, int b,
                                           int lane) {
    const int rb0 = p.rb_first + c * p.R, n = min(nb - rb0, p.R);
    if (lane == 0) mbar_expect_tx(st.bar + b, (unsigned)(n * p.W * 256));
    __syncwarp();
    if (lane < n)
        bulk_g2s(st.buf + b * st.stride + lane * p.W * 32, op + (size_t)(tri_frags(rb0 + lane) + p.klo) * 32, (unsigned)(p.W * 256),
                 st.bar + b);
}
// row blocks [rb0, rb1) of a slab chunk that starts at row block rb0 (register tile: see row_blocks_rolled)
template <int KS, int NT, int TABN, bool REL>
__device__ __forceinline__ void slab_rows(const double *buf, const SlabPlan &p, int rb0, int rb1, double (&bf)[KS][NT],
                                          double (&q0)[NT], double (&q1)[NT], typename KMask<KS>::type mask, int lane, int k0,
                                          const Wide<NT> &w) {
    if constexpr (REL) {
        if (w.on) {
            const int kfirst = __ffsll((long long)w.mask) - 1;
#pragma unroll 1
            for (int rb = max(rb0, kfirst >> 1); rb < rb1; ++rb)
                wide_row_block<KS, NT, TABN>(buf + ((rb - rb0) * p.W - p.klo) * 32 + lane, 2 * rb + 2, w, bf, q0, q1);
            return;
        }
    }
    if (!mask) return;
    int g0, kend;
    mask_groups(mask, g0, kend);
    const int kfirst = k0 + __ffsll((long long)(unsigned long long)mask) - 1;
    int rb = rb0;
    const bool rect = REL && plain_band(mask, g0, kend);
    const int kend2 = (64 - __clzll((long long)(unsigned long long)mask) + 1) & ~1;
    const int rbf = rect ? min(rb1, max(rb0, ((k0 + kend2) >> 1) & ~1)) : rb1;
#pragma unroll 1
    for (; rb + 1 < rbf; rb += 2) {
        if (2 * rb + 4 <= kfirst) continue;
        const double *afA = buf + ((rb - rb0) * p.W - p.klo + k0) * 32 + lane;       // afA[j * 32] = fragment (rb, k0 + j)
        if (REL && rect) row_block_pair<KS, NT, REL>(afA, afA + p.W * 32, 2 * rb + 2 - k0, bf, q0, q1, mask, g0, kend);
        else row_block_pair<KS, NT>(afA, afA + p.W * 32, 2 * rb + 2 - k0, bf, q0, q1, mask, g0, kend);
    }
    if constexpr (REL) {
        if (rect && rb + 1 < rb1) {
            const int npair = (rb1 - rb) >> 1;
            rect_dispatch<KS, NT>(kend2 >> 1, buf + ((rb - rb0) * p.W - p.klo + k0) * 32 + lane, npair, p.W * 32, 2 * p.W * 32, 0, 0, bf, q0,
                                  q1);
            rb += 2 * npair;
        }
    }
    if (rb < rb1) row_block<KS, NT>(buf + ((rb - rb0) * p.W - p.klo + k0) * 32 + lane, 2 * rb + 2 - k0, bf, q0, q1, mask);
}
// The DMMAs of one operand for one sub-tile.  `res`: the whole slab already sits in the (contiguous) buffers, fetched once
// per super-tile on barrier 0 -- the first sub-tile waits for it.  Otherwise the slab is streamed for this sub-tile in
// chunks: chunks 0 and 1 were issued by the caller, chunk c lives in buffer c & 1 and chunk c + 2 is issued once every
// warp is done with chunk c.
template <int KS, int NT, int TABN, bool REL>
__device__ __forceinline__ void slab_pass(const double *__restrict__ op, const SlabPlan &p, bool res, bool first_sub, Stream &st,
                                          double (&bf)[KS][NT], double (&q0)[NT], double (&q1)[NT], int nb, int lane, int warp,
                                          typename KMask<KS>::type mask, int k0, const Wide<NT> &w) {
    const int nch = res ? (p.nchunk ? 1 : 0) : p.nchunk;
    const int R = res ? nb - p.rb_first : p.R;
#pragma unroll 1
    for (int c = 0; c < nch; ++c) {
        const int b = res ? 0 : (c & 1);
        if (!res || first_sub) {
            mbar_wait(st.bar + b, (st.phase >> b) & 1u);        // the chunk (slab) has landed
            st.phase ^= 1u << b;
        }
        const int rb0 = p.rb_first + c * R;
        slab_rows<KS, NT, TABN, REL>(st.buf + b * st.stride, p, rb0, min(nb, rb0 + R), bf, q0, q1, mask, lane, k0, w);
        if (!res) {
            __syncthreads();                                    // every warp is done with buffer b
            if (warp == 0 && c + 2 < nch) slab_issue(op, p, c + 2, nb, st, b, lane);
        }
    }
}

// Dense candidate / g rows of one dense row block: acc += A(db, k0 + j) . bf[j] over the relevant exp groups of the (relative)
// mask.  af[j * 32] = fragment (db, k0 + j); nk = k-steps that exist from the tile start on (fragments past it are not read).
template <int KB, int NT, int GK = exp_group<NT>()>
__device__ __forceinline__ void dense_acc(const double *af, int nk, const double (&bf)[KB][NT], typename KMask<KB>::type mask,
                                          double (&c0)[NT], double (&c1)[NT], double (&e0)[NT], double (&e1)[NT]) {
    using mask_t = typename KMask<KB>::type;       // GK: the groups of gen_exps -- all of a relevant group's B fragments exist
#pragma unroll
    for (int g = 0; g < KB / GK; ++g) {
        if ((mask >> (GK * g)) & (((mask_t)1 << GK) - 1)) {     // warp-uniform: a real branch around GK DMMAs
            double fa[GK];
#pragma unroll
            for (int j = 0; j < GK; ++j) fa[j] = (GK * g + j < nk) ? af[(GK * g + j) * 32] : 0.0;
#pragma unroll
            for (int j = 0; j < GK; j += 2)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    dmma(c0[nt], c1[nt], fa[j], bf[GK * g + j][nt]);
                    dmma(e0[nt], e1[nt], fa[j + 1], bf[GK * g + j + 1][nt]);     // 2 chains: the dense rows are few
                }
        }
    }
}

// Sum the 8 row slots of the squared accumulators (lanes with equal lane & 3) and park them in scratch row `row`
template <int NT>
__device__ __forceinline__ void park_q(double (&q0)[NT], double (&q1)[NT], double *scr, int row, int col0, int kq, int pq) {
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
#pragma unroll
        for (int o = 4; o < 32; o <<= 1) {
            q0[nt] += __shfl_xor_sync(0xffffffffu, q0[nt], o);
            q1[nt] += __shfl_xor_sync(0xffffffffu, q1[nt], o);
        }
        if (pq == 0) *reinterpret_cast<double2 *>(scr + row * SCR_STRIDE + col0 + nt * 8 + 2 * kq) = make_double2(q0[nt], q1[nt]);
    }
}

// MODE 0: esm / em / status.  MODE 1: additionally the fused expected-variance + argmin epilogue.  MODE 2: prediction --
// the same passes, but the tail returns the posterior mean of gp_l (BQ.l_mean, bq.py:177-200) in `esm` and the
// posterior variance of gp_log_l (the factor of BQ.l_var, bq.py:202-231) in `em`: no shortcut, no jitter pattern.
// BK > 0: band-relative register tile of BK k-steps (see row_blocks_rolled); BK = 0: the tile covers all KS k-steps.
template <int KS, int NT, int WARPS, int MINB, bool STREAM, int TABN, int ALIGN, bool ROLLED, int BK, int MODE>
__global__ void __launch_bounds__(WARPS * 32, MINB) bq_score_kernel(ScoreArgs a) {
    constexpr bool EPI = MODE == 1, PRED = MODE == 2;
    constexpr bool REL = BK > 0;
    constexpr int KB = REL ? BK : KS;                       // k-steps of the register tile
    static_assert(!REL || (BK % 8 == 0 && BK <= KS), "band tile: whole exp groups, no larger than the class");
    using rmask_t = typename KMask<KB>::type;
    // exp groups of the fast path: with 16 warps per SM the latency of four chains is covered by the other warps, and a band
    // of 8-14 k-steps wastes fewer exponentials on groups of 4 than on groups of 8
    constexpr int GKK = REL ? BQB_REL_GK : exp_group<NT>();
    using SM = ScoreSmem<KS, NT, WARPS, STREAM, TABN>;
    constexpr bool LOCKSTEP = STREAM || ALIGN != 0;         // warps must keep reaching the barriers
    static_assert(ALIGN <= 1 || WARPS % ALIGN == 0, "barrier groups of whole warps");
    constexpr int THREADS = WARPS * 32;
    constexpr int SUB = 4 / NT;                             // sub-tiles of 8 NT points per 32-point super-tile
    extern __shared__ __align__(16) double smem[];
    const Layout lay = a.lay;
    __shared__ __align__(16) double s_tab[TABN];            // static: its address is an immediate of every table LDS
    double *s_small = smem;
    double *s_ops = s_small + lay.n_small;                  // resident operands, or the two chunk buffers + dense rows
    double *s_af_l = s_ops;
    // Shared memory is sized for what the launch's instances need (row blocks, dense rows) in the large classes; the
    // ns <= 64 kernels sit at their register limit and keep the class maxima as compile-time constants.
    constexpr bool RT_SIZES = KS > 16;
    const int nb_res = RT_SIZES ? a.nb_res : KS / 2, nrow_res = RT_SIZES ? a.nrow_res : 8 * a.ndb_max;
    double *s_af_d = STREAM ? s_ops + 2 * a.chunk_frags * 32 : s_af_l + tri_frags(nb_res) * 32;
    double *s_af_t = s_af_d + a.ndb_max * 2 * nb_res * 32;            // (resident only)
    double *s_scr = s_ops + SM::operands(a.ndb_max, a.chunk_frags, nb_res);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int inst = a.inst0 + blockIdx.y;
    const double *M = a.models + (size_t)inst * lay.total;

    __shared__ int s_cta_st;                                // OR of the status bits of this CTA's points (a.cta_flags)
    if (tid == 0) s_cta_st = 0;
    for (int i = tid; i < TABN; i += THREADS) s_tab[i] = a.exp_tab[(TABN == 2048 ? 0 : 2048) + i];
    for (int i = tid; i < lay.n_small; i += THREADS) s_small[i] = M[i];
    __syncthreads();
    const int nc = (int)s_small[H_NC], nsp = (int)s_small[H_NSP], ndb = (int)s_small[H_NDB];
    const int nb = nsp >> 3, nks = nsp >> 2;
    __shared__ __align__(8) unsigned long long s_bar[2];
    // the warps' relevance masks (K_l, K_tl) of a sub-tile; two sets alternate so that a fast warp's next sub-tile cannot
    // overwrite what a slow warp still reads (there is no CTA barrier between two sub-tiles that stream nothing)
    __shared__ unsigned long long s_wm[STREAM ? 4 * WARPS : 1];
    int wm_set = 0;
    Stream strm{s_bar, s_ops, a.chunk_frags * 32, 0u};
    if constexpr (STREAM) {
        if (tid == 0) {
            mbar_init(s_bar, 1);
            mbar_init(s_bar + 1, 1);
            mbar_init_fence();
        }
    } else {
        stage<THREADS>(s_af_l, M + lay.off_af_l_tri, tri_frags(nb) * 32);
        stage<THREADS>(s_af_t, M + lay.off_af_tl_tri, tri_frags(nb) * 32);
    }
    stage<THREADS>(s_af_d, M + lay.off_af_l_dense, ndb * nks * 32);     // the dense rows are resident in both variants
    __syncthreads();

    const double *s_xs = s_small + lay.off_xs, *s_tol = s_small + lay.off_tol, *s_atl = s_small + lay.off_atl;
    const double nhl = s_small[H_NHL];
    const double Cl = nhl * ExpC<TABN>::INVN, Ctl = s_small[H_NHTL] * ExpC<TABN>::INVN;   // exponent scale in table units
    const int dmax_l = exp_d2max_hi(nhl), dmax_tl = exp_d2max_hi(s_small[H_NHTL]);
    using mask_t = typename KMask<KS>::type;
    // relevance threshold in units of d^2 (a.cut_arg = CUT_ARG, or +inf: every k-step is relevant, the dense algorithm)
    const double cut_l = a.cut_arg / fabs(nhl), cut_tl = a.cut_arg / fabs(s_small[H_NHTL]);
    unsigned long long n_kstep = 0;                         // (row block, k-step) products executed by this warp (a.work)
    const int tol2_hi = __double2hiint(s_small[H_TOL2MAX]) + 1;
    double *scr = s_scr + warp * SM::scr(nrow_res);        // rows: 0 qs, 1 qt, 2 tm, 3 isclose, 4.. dense rows, then x_a

    const double *xa = a.x_a + (size_t)(inst / a.xa_group) * a.xa_stride;
    double *o_esm = a.esm ? a.esm + (size_t)inst * a.out_stride : nullptr;   // optional when the fused epilogue writes ev
    double *o_em = a.em ? a.em + (size_t)inst * a.out_stride : nullptr;
    int *o_st = a.status ? a.status + (size_t)inst * a.out_stride : nullptr;

    const int kq = lane & 3, pq = lane >> 2;
    // Work distribution.  A UNIT is 8 NT WARPS points (one sub-tile per warp), a super-tile SUB units (32 points per
    // warp).  Whole super-tiles are dealt round-robin (tile it * G + c to CTA c: expensive neighbourhoods -- points
    // close to a candidate refactorise the Schur block in the tail -- are spread over all CTAs; contiguous runs per CTA
    // measured 12 % slower on C2), every CTA taking the same number `full` of them; the remaining R < G SUB units are
    // split evenly at unit granularity, so a CTA ends with one partial super-tile of r_n < SUB units (8 NT r_n points
    // per warp).  With whole super-tiles only, the last of the ~14 rounds of a 10^6-point launch was 80 % idle.
    constexpr int UNIT = 8 * NT * WARPS;
    const int n_units = (a.na + UNIT - 1) / UNIT;
    const int G = gridDim.x, cta = blockIdx.x;
    const int full = n_units / (G * SUB);
    const int R = n_units - full * G * SUB;
    const int r_lo = full * G * SUB + (int)(((long long)cta * R) / G);
    const int r_n = (int)(((long long)(cta + 1) * R) / G) - (int)(((long long)cta * R) / G);
    const int n_it = full + (r_n > 0 ? 1 : 0);
    auto tile_u = [&](int it) { return it < full ? (it * G + cta) * SUB : r_lo; };       // first unit of tile `it`
    auto tile_n = [&](int it) { return it < full ? SUB : r_n; };                         // its units
    double best_v = INFINITY;                               // fused argmin of ev: this lane's running (min, first index)
    long long best_i = 0x7fffffffffffffffLL;

    int xb = 0;                                             // xrows + 32 xb holds this super-tile's points
    double *xrows = scr + (SCR_DENSE + nrow_res) * SCR_STRIDE;        // two 32-point rows
    if (n_it > 0) fetch_points(xrows, xa, (long long)tile_u(0) * UNIT + warp * (8 * NT * tile_n(0)), a.na, lane);
    async_commit();

    for (int it = 0; it < n_it; ++it) {
        const int nsub = tile_n(it);                 // units (= sub-tiles per warp) of this super-tile
        const int npw = 8 * NT * nsub;               // points per warp
        const int base = tile_u(it) * UNIT + warp * npw;
        const double *xrow = xrows + 32 * xb;
        async_wait<0>();                             // this super-tile's points have landed (fetched one tile ago) ...
        __syncwarp();                                // ... for every lane of the warp
        xb ^= 1;
        if (it + 1 < n_it)
            fetch_points(xrows + 32 * xb, xa, (long long)tile_u(it + 1) * UNIT + warp * (8 * NT * tile_n(it + 1)), a.na, lane);
        async_commit();
        if (!LOCKSTEP && base >= a.na) continue;     // warp-uniform; lock-step warps must keep hitting the barriers

        // ---- STREAM: what to stream for this super-tile.  Relevance masks of all its sub-tiles (a cheap extra distance
        // pass) are OR-ed over the CTA; if the resulting band slab of an operand fits the two chunk buffers it is fetched
        // ONCE and serves every sub-tile (pass-major order: K_l for all sub-tiles, then K_tl), otherwise each sub-tile
        // streams it in chunks.
        // relevance masks of this warp's points (both kernels; shared by the super-tile's sub-tiles)
        mask_t wmask_l, wmask_tl;
        {
            const double xv = xrow[lane];
            gen_masks<KS>(xv, lane < npw && base + lane < a.na && isfinite(xv), cut_l, cut_tl, nsp, lane, s_xs, wmask_l, wmask_tl);
        }
        // ---- STREAM: what to stream for this super-tile.  The warps' masks are OR-ed over the CTA; if the resulting band
        // slab of an operand fits the two chunk buffers it is fetched ONCE and serves every sub-tile (pass-major order: K_l
        // for all sub-tiles, then K_tl), otherwise each sub-tile streams it in chunks.
        SlabPlan plan_l, plan_tl;
        bool res_l = false, res_tl = false;
        if constexpr (STREAM) {
            unsigned long long *wm = s_wm + wm_set * 2 * WARPS;
            wm_set ^= 1;
            if (lane == 0) { wm[2 * warp] = wmask_l; wm[2 * warp + 1] = wmask_tl; }
            __syncthreads();                             // (every warp has also left the previous super-tile's buffers)
            unsigned long long um_l = 0, um_tl = 0;
#pragma unroll
            for (int w = 0; w < WARPS; ++w) { um_l |= wm[2 * w]; um_tl |= wm[2 * w + 1]; }
            plan_l = make_slab_plan<KS>((mask_t)um_l, nks, nb, a.chunk_frags);
            plan_tl = make_slab_plan<KS>((mask_t)um_tl, nks, nb, a.chunk_frags);
            res_l = (nb - plan_l.rb_first) * plan_l.W <= 2 * a.chunk_frags;
            res_tl = (nb - plan_tl.rb_first) * plan_tl.W <= 2 * a.chunk_frags;
        }

        // band-relative tile: where this warp's band starts in each kernel, and whether it fits the register tile
        int k0_l = 0, k0_tl = 0;
        Wide<NT> wd_l, wd_tl;
        wd_l.on = wd_tl.on = false;
        if constexpr (REL) {
            auto band = [&](mask_t m, int &k0, Wide<NT> &w, double C, int dmax) {
                w.mask = m; w.C = C; w.dmax = dmax; w.kq = lane & 3; w.s_xs = s_xs; w.s_tab = s_tab;
                w.kbeg = w.kend = 0;
                if (!m) return;
                const int lo = __ffsll((long long)(unsigned long long)m) - 1, hi = 64 - __clzll((long long)(unsigned long long)m);
                w.kbeg = lo & ~7; w.kend = hi;                    // wide path: windows from a whole exp group
                // fast path: the band fits the tile and has no holes (sorted observations and the interval criterion of
                // gen_masks give contiguous masks; anything else is walked pair by pair on the wide path, which never
                // touches a fragment outside [lo & ~1, hi + 1) -- all a slab holds)
                const unsigned long long mb = (unsigned long long)m >> lo;
                w.on = (hi - (lo & ~1) > KB) || (mb & (mb + 1)) != 0 || a.force_wide;
                k0 = w.on ? 0 : (lo & ~1);                        // even: row blocks end on even k-steps; the band starts in group 0
            };
            band(wmask_l, k0_l, wd_l, Cl, dmax_l);
            band(wmask_tl, k0_tl, wd_tl, Ctl, dmax_tl);
        }

        constexpr int NPH = STREAM ? 2 : 1;              // STREAM: pass 0 = K_l, pass 1 = K_tl; otherwise both per sub-tile
#pragma unroll
        for (int ph = 0; ph < NPH; ++ph) {
            const bool do_l = !STREAM || ph == 0, do_tl = !STREAM || ph == 1;
            const SlabPlan &plan = ph ? plan_tl : plan_l;
            const bool res = ph ? res_tl : res_l;
            const double *op = M + (ph ? lay.off_af_tl_tri : lay.off_af_l_tri);
            if constexpr (STREAM) {
                if (ph == 1) __syncthreads();            // every warp is done with the K_l slab
                if (res && plan.nchunk && warp == 0) {   // whole slab: one copy per row block, all on barrier 0
                    const int n = nb - plan.rb_first;
                    if (lane == 0) mbar_expect_tx(strm.bar, (unsigned)(n * plan.W * 256));
                    __syncwarp();
                    if (lane < n)
                        bulk_g2s(strm.buf + lane * plan.W * 32, op + (size_t)(tri_frags(plan.rb_first + lane) + plan.klo) * 32,
                                 (unsigned)(plan.W * 256), strm.bar);
                }
            }
#pragma unroll 1
            for (int sub = 0; sub < nsub; ++sub) {
                const int col0 = sub * 8 * NT;
                double x[NT];
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    const double v = xrow[col0 + nt * 8 + pq];      // points past na were filled with 0
                    x[nt] = isfinite(v) ? v : 0.0;       // invalid x_a is reported by the tail (ST_XA_BAD)
                }
                double bf[KB][NT];
                double q0[NT], q1[NT], tm[NT];
                int close[NT];
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) { q0[nt] = q1[nt] = tm[nt] = 0.0; close[nt] = 0; }
                mask_t mask = wmask_l;
                const mask_t mask_tl = wmask_tl;
                if constexpr (REL) {
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) wd_l.x[nt] = wd_tl.x[nt] = x[nt];
                }
                if constexpr (STREAM) {
                    if (!res && plan.nchunk && warp == 0) {                 // chunked: first two chunks, under the exp phase
                        slab_issue(op, plan, 0, nb, strm, 0, lane);
                        if (plan.nchunk > 1) slab_issue(op, plan, 1, nb, strm, 1, lane);
                    }
                }

                if (do_l) {
                    // ---- K_l: cross-kernel fragments, triangular rows then the dense candidate / g rows
                    phase_sync<ALIGN>();                 // enter the exp phase together (DMMA / DFMA mixing costs pipe throughput)
                    // relative mask of the register tile (empty on the wide path, which generates its windows itself)
                    const rmask_t rm_l = REL ? (wd_l.on ? (rmask_t)0 : (rmask_t)(mask >> k0_l)) : (rmask_t)mask;
                    gen_exps<KB, NT, TABN, false, GKK>(bf, x, Cl, dmax_l, rm_l, kq, s_xs + 4 * k0_l, s_atl, s_tab, tm, tol2_hi, close);
                    if constexpr (STREAM)
                        slab_pass<KB, NT, TABN, REL>(op, plan, res, sub == 0, strm, bf, q0, q1, nb, lane, warp, rm_l, k0_l, wd_l);
                    else tri_pass<KB, NT, TABN, ALIGN, ROLLED, REL>(s_af_l, bf, q0, q1, nb, lane, rm_l, k0_l, wd_l);
                    if (a.work) n_kstep += count_ksteps<KS>(mask, nb) + ndb * __popcll((unsigned long long)mask);
#pragma unroll
                    for (int db = 0; db < 3; ++db) {
                        if (db < ndb) {
                            const double *af = s_af_d + (db * nks) * 32 + lane;
                            double c0[NT], c1[NT], e0[NT], e1[NT];
#pragma unroll
                            for (int nt = 0; nt < NT; ++nt) { c0[nt] = c1[nt] = e0[nt] = e1[nt] = 0.0; }
                            if (REL && wd_l.on) {                          // wide band: window by window (exponentials regenerated)
#pragma unroll 1
                                for (int kw = wd_l.kbeg; kw < wd_l.kend; kw += KB) {
                                    const rmask_t rw = window_mask<KB>(wd_l.mask, kw);
                                    if (!rw) continue;
                                    gen_exps<KB, NT, TABN, false>(bf, x, Cl, dmax_l, rw, kq, s_xs + 4 * kw, s_atl, s_tab, tm, tol2_hi, close);
                                    dense_acc<KB, NT>(af + kw * 32, nks - kw, bf, rw, c0, c1, e0, e1);
                                }
                            } else {
                                dense_acc<KB, NT, GKK>(af + k0_l * 32, nks - k0_l, bf, rm_l, c0, c1, e0, e1);
                            }
                            if (!RT_SIZES || db * 8 + pq < nrow_res) {      // only the nc + 2 rows that exist have a scratch row
#pragma unroll
                                for (int nt = 0; nt < NT; ++nt)
                                    *reinterpret_cast<double2 *>(scr + (SCR_DENSE + db * 8 + pq) * SCR_STRIDE + col0 + nt * 8 + 2 * kq) =
                                        make_double2(c0[nt] + e0[nt], c1[nt] + e1[nt]);
                            }
                        }
                    }
                    park_q<NT>(q0, q1, scr, 0, col0, kq, pq);
                }

                if (do_tl) {
                    // ---- K_tl: fragments, gp_log_l.mean and the isclose test
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) { q0[nt] = q1[nt] = 0.0; }
                    phase_sync<ALIGN>();
                    mask = mask_tl;
                    const rmask_t rm_tl = REL ? (wd_tl.on ? (rmask_t)0 : (rmask_t)(mask >> k0_tl)) : (rmask_t)mask;
                    if (REL && wd_tl.on) {                   // wide band: gp_log_l.mean and the isclose pre-filter, window by window
#pragma unroll 1
                        for (int kw = wd_tl.kbeg; kw < wd_tl.kend; kw += KB) {
                            const rmask_t rw = window_mask<KB>(wd_tl.mask, kw);
                            if (!rw) continue;
                            int cw[NT];
                            gen_exps<KB, NT, TABN, true>(bf, x, Ctl, dmax_tl, rw, kq, s_xs + 4 * kw, s_atl + 4 * kw, s_tab, tm, tol2_hi, cw,
                                                         KS - kw);
#pragma unroll
                            for (int nt = 0; nt < NT; ++nt) close[nt] |= cw[nt];
                        }
                    } else {
                        gen_exps<KB, NT, TABN, true, GKK>(bf, x, Ctl, dmax_tl, rm_tl, kq, s_xs + 4 * k0_tl, s_atl + 4 * k0_tl, s_tab, tm,
                                                          tol2_hi, close, KS - k0_tl);
                    }
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt)
                        if (close[nt]) close[nt] = isclose_exact(x[nt], s_xs, s_tol, nsp, kq);
                    if constexpr (STREAM)
                        slab_pass<KB, NT, TABN, REL>(op, plan, res, sub == 0, strm, bf, q0, q1, nb, lane, warp, rm_tl, k0_tl, wd_tl);
                    else tri_pass<KB, NT, TABN, ALIGN, ROLLED, REL>(s_af_t, bf, q0, q1, nb, lane, rm_tl, k0_tl, wd_tl);
                    if (a.work) n_kstep += count_ksteps<KS>(mask, nb);
                    park_q<NT>(q0, q1, scr, 1, col0, kq, pq);
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        tm[nt] += __shfl_xor_sync(0xffffffffu, tm[nt], 1);
                        tm[nt] += __shfl_xor_sync(0xffffffffu, tm[nt], 2);
                        close[nt] |= __shfl_xor_sync(0xffffffffu, close[nt], 1);
                        close[nt] |= __shfl_xor_sync(0xffffffffu, close[nt], 2);
                        if (kq == 0) {
                            scr[2 * SCR_STRIDE + col0 + nt * 8 + pq] = tm[nt];
                            scr[3 * SCR_STRIDE + col0 + nt * 8 + pq] = close[nt] ? 1.0 : 0.0;
                        }
                    }
                }
            }
        }
        __syncwarp();

        // ================= tail: one lane per point of the super-tile
        const int p = base + lane;
        if (lane < npw && p < a.na) {
            const double xv = xrow[lane];
            const double Zm = s_small[H_ZM];
            double esm, em;
            int st = ST_OK;
            if (!isfinite(xv)) {
                esm = em = nan("");
                st = ST_XA_BAD;
            } else if (!PRED && scr[3 * SCR_STRIDE + lane] != 0.0) {
                em = Zm; esm = Zm * Zm; st = ST_SHORTCUT;         // bq.py:456-459
            } else {
                const double qs = scr[lane], qt = scr[SCR_STRIDE + lane], tmv = scr[2 * SCR_STRIDE + lane];
                double *dr = scr + SCR_DENSE * SCR_STRIDE + lane;          // dense row r at dr[r * SCR_STRIDE]; reused for v_c
                const double c_l = s_small[H_CL], thresh = s_small[H_THRESH];
                const double *s_xc = s_small + lay.off_xc;
                unsigned mask = 0;
                for (int j = 0; j < nc; ++j) {
                    const double dc = s_xc[j] - xv;
                    if (!PRED && fabs(dc) < thresh) mask |= 1u << j;     // bq.py:470 (strict <)
                    dr[j * SCR_STRIDE] = fma(c_l, exp_kernel<TABN>(dc * dc, Cl, dmax_l, s_tab), dr[j * SCR_STRIDE]);   // w = k_c + W k_s
                }
                double qc = 0, vg = 0, va = 0, bg = 0, kaa;     // bg = u_gamma_c . u_alpha_c of this pattern
                bool pd = true;
                if (mask == 0) {
                    const double *Lc = s_small + lay.off_lcc0, *ug = s_small + lay.off_ug0, *ua = s_small + lay.off_ua0,
                                 *rd = s_small + lay.off_rd0;
                    for (int i = 0; i < nc; ++i) {
                        double s = dr[i * SCR_STRIDE];
                        for (int k = 0; k < i; ++k) s = fma(-Lc[i * NC_MAX + k], dr[k * SCR_STRIDE], s);
                        s *= rd[i];
                        dr[i * SCR_STRIDE] = s;
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
                            double s = dr[i * SCR_STRIDE], sg = wb[i], sa = wa[i];
                            for (int k = 0; k < i; ++k) {
                                const double l = Lc[i * (i + 1) / 2 + k];
                                s -= l * dr[k * SCR_STRIDE]; sg -= l * ug[k]; sa -= l * ua[k];
                            }
                            const double d = Lc[i * (i + 1) / 2 + i];
                            s /= d; sg /= d; sa /= d;
                            dr[i * SCR_STRIDE] = s; ug[i] = sg; ua[i] = sa;
                            qc = fma(s, s, qc); vg = fma(s, sg, vg); va = fma(s, sa, va);
                            bg = fma(sg, sa, bg);
                        }
                    }
                    kaa = s_small[H_KAA_N];
                }
                const double s_ = kaa - (qs + qc);                        // Schur pivot of the new point
                if (PRED) {
                    esm = dr[(nc + 1) * SCR_STRIDE] + va;                 // gp_l.mean(x) = K_l(x, x_sc) alpha_l
                    em = s_small[H_KTT] - qt;                             // diag gp_log_l.cov(x)
                } else if (!pd || !(s_ > 0.0)) {
                    em = Zm; esm = Zm * Zm; st = ST_NOTPD;                // bq.py:481-490
                } else {
                    const double ba = s_small[H_BA_S] + bg;               // int_K(x_sc) . alpha_P
                    const double kg = dr[nc * SCR_STRIDE] + vg;           // k_a . gamma_P
                    const double ka = dr[(nc + 1) * SCR_STRIDE] + va;     // k_a . alpha_P
                    // int_K at the new point (gauss_c.pyx:162): h^2 N(x_a | mu, w_l^2 + sigma^2)
                    const double diff = xv - s_small[H_MU];
                    const double b_a = s_small[H_CB] * exp_tab<TABN>((diff * diff) * s_small[H_NHB], s_tab);
                    const double A_a = (b_a - kg) / s_;                   // last entry of K_sca^-1 int_K (bq_c.pyx:467-469)
                    const double A_sc_l = ba - A_a * ka;                  // dot(A_sca[:-1], l_sc)       (bq_c.pyx:470)
                    const double tC = s_small[H_KTT] - qt;                // gp_log_l.cov(x_a)            bq.py:496
                    const double a1 = tmv + 0.5 * tC;                     // int_exp_norm(1, tm, tC)      gauss_c.pyx:87
                    const double a2 = 2.0 * tmv + 2.0 * tC;               // int_exp_norm(2, tm, tC)
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
            const int po = a.perm ? a.perm[p] : p;          // the point's position in the caller's (unsorted) vector
            if (o_esm) o_esm[po] = esm;
            if (EPI) {
                const double evv = __dsub_rn(__dadd_rn(__dmul_rn(Zm, Zm), s_small[H_ZV]), esm);   // no FMA contraction: matches the host
                a.ev[po] = evv;
                if (evv < best_v || (evv == best_v && po < best_i)) { best_v = evv; best_i = po; }   // ties keep the first index
            }
            if (o_em) o_em[po] = em;
            if (o_st) o_st[po] = st;
            if (st) {                                       // rare: shortcut / fallback / invalid points
                if (a.flags) atomicOr(a.flags + inst, st);
                if (a.cta_flags) atomicOr(&s_cta_st, st);
            }
        }
        __syncwarp();
    }
    if (a.work && lane == 0 && n_kstep) atomicAdd(a.work, n_kstep * NT);     // DMMA instructions of this warp
    if (a.cta_flags) {                                      // one plain store per CTA (the array may be page-locked host memory)
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
        __syncthreads();                                    // scratch is free: every warp has left the tile loop
        double *rv = s_scr;
        long long *ri = reinterpret_cast<long long *>(s_scr + WARPS);
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

#ifndef BQB_REL_DEFAULT
#define BQB_REL_DEFAULT 1
#endif
constexpr size_t SMEM_LIMIT = 227 * 1024;      // per-CTA opt-in maximum on sm_100 (static + dynamic)
constexpr size_t SMEM_STATIC_MISC = 256;       // chunk table, mbarriers

// Row blocks the resident operands are sized for / dense rows kept in scratch: what the launch's instances need (set by
// the C-ABI layer from the batch's counts), or the class maximum when unknown
template <int KS>
static int res_rows(const ScoreArgs &a) { return (KS > 16 && a.nb_max > 0 && a.nb_max < KS / 2) ? a.nb_max : KS / 2; }
template <int KS>
static int dense_rows(const ScoreArgs &a) {
    return (KS > 16 && a.nrow_max > 0 && a.nrow_max < 8 * a.ndb_max) ? a.nrow_max : 8 * a.ndb_max;
}

// Bytes of shared memory (static + dynamic) an instantiation needs for this launch
template <int KS, int NT, int WARPS, bool STREAM, int TABN>
static size_t smem_need(const ScoreArgs &a, int chunk_frags) {
    return sizeof(double) * (TABN + ScoreSmem<KS, NT, WARPS, STREAM, TABN>::doubles(a.lay.n_small, a.ndb_max, chunk_frags,
                                                                                    res_rows<KS>(a), dense_rows<KS>(a))) +
           SMEM_STATIC_MISC;
}

template <int KS, int NT, int WARPS, int MINB, bool STREAM, int TABN, int ALIGN, bool ROLLED, int BK, int MODE>
static cudaError_t launch_cfg2(ScoreArgs a, int n_inst, int sm_count, cudaStream_t stream, int *grid_x) {
    using SM = ScoreSmem<KS, NT, WARPS, STREAM, TABN>;
    a.chunk_frags = 0;
    a.nb_res = res_rows<KS>(a);
    a.nrow_res = dense_rows<KS>(a);
    if (STREAM) {       // the largest chunk buffers that fit
        int cf = CHUNK_FRAGS_MAX;
        while (cf >= 2 * KS && smem_need<KS, NT, WARPS, STREAM, TABN>(a, cf) > SMEM_LIMIT) cf -= 16;
        if (cf < 2 * KS) return cudaErrorInvalidConfiguration;      // a slab chunk holds at least two whole row blocks
        a.chunk_frags = cf;
    }
    const size_t bytes = sizeof(double) * SM::doubles(a.lay.n_small, a.ndb_max, a.chunk_frags, a.nb_res, a.nrow_res);
    auto kern = bq_score_kernel<KS, NT, WARPS, MINB, STREAM, TABN, ALIGN, ROLLED, BK, MODE>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return e;
    const int n_units = (a.na + 8 * NT * WARPS - 1) / (8 * NT * WARPS);
    // persistent: at most MINB CTAs per SM in total.  Rounding the share of an instance UP (the round-1 rule) put e.g. 64
    // instances x 5 CTAs = 320 CTAs on 296 slots: a second wave of 24 CTAs that doubled the launch's duration.  With fewer
    // instances than slots every instance gets floor(slots / n_inst) CTAs (one wave); with more, one CTA each.
    int per_inst = (sm_count * MINB) / n_inst;
    if (per_inst > n_units) per_inst = n_units;
    if (per_inst < 1) per_inst = 1;
    dim3 grid(per_inst, n_inst);
    if (grid_x) *grid_x = per_inst;
    kern<<<grid, WARPS * 32, bytes, stream>>>(a);
    return cudaGetLastError();
}

template <int KS, int NT, int WARPS, int MINB, bool STREAM, int TABN, int ALIGN, bool ROLLED, int BK = 0>
static cudaError_t launch_cfg(const ScoreArgs &a, int n_inst, int sm_count, cudaStream_t stream, int *grid_x) {
    // the fused expected-variance / argmin epilogue is a separate instantiation so that plain scoring keeps its registers
    if (a.predict) return launch_cfg2<KS, NT, WARPS, MINB, STREAM, TABN, ALIGN, ROLLED, BK, 2>(a, n_inst, sm_count, stream, grid_x);
    if (a.ev) return launch_cfg2<KS, NT, WARPS, MINB, STREAM, TABN, ALIGN, ROLLED, BK, 1>(a, n_inst, sm_count, stream, grid_x);
    return launch_cfg2<KS, NT, WARPS, MINB, STREAM, TABN, ALIGN, ROLLED, BK, 0>(a, n_inst, sm_count, stream, grid_x);
}

// Kernel choice of the large classes (environment, read at every launch): BQB_REL = 1 (default) band-relative register tile
// of 24 k-steps with 16 warps per CTA, 0 the absolute tile with 8 warps (the previous kernels, kept for A/B runs and as the
// cross-check of tests/test_gpu_parity.py).  12 warps at 166 registers measured the same at ns = 128 and 7 % slower at
// ns = 256.  BQB_FORCE_WIDE = 1 sends every warp down the wide path (tests).
[[maybe_unused]] static int rel_variant() {
    const char *e = getenv("BQB_REL");
    return e ? atoi(e) : BQB_REL_DEFAULT;
}
[[maybe_unused]] static ScoreArgs with_env(ScoreArgs a) {
    const char *e = getenv("BQB_FORCE_WIDE");
    a.force_wide = (e && atoi(e)) ? 1 : 0;
    return a;
}

// nsp_cap selects the instantiation: 16, 64, 128 (operands resident), 160 and 256 (operands streamed).  The tilings
// are the measured best of the round-1 sweeps (profiles/ncu_score_r01.md); a resident instantiation falls back to the
// streamed one when many candidates (scratch rows) push it over the shared-memory limit.
//
// This file is compiled once per capacity class (-DBQB_SCORE_CLASS=16|64|128|160|256: the instantiations of that class
// only, so that the classes build in parallel) and once without the macro (the dispatcher).
#define BQB_LAUNCH_DECL(C) cudaError_t launch_score_##C(const ScoreArgs &a, int n_inst, int sm_count, cudaStream_t stream, int *grid_x)
// band-relative kernels of a class: a translation unit of their own (-DBQB_SCORE_REL=1) so that the build stays parallel;
// returns cudaErrorInvalidConfiguration, without launching, when their shared memory does not fit this launch
#define BQB_LAUNCH_REL_DECL(C) cudaError_t launch_score_rel_##C(const ScoreArgs &a, int n_inst, int sm_count, cudaStream_t stream, int *grid_x)
#ifndef BQB_SCORE_CLASS
BQB_LAUNCH_DECL(16);
BQB_LAUNCH_DECL(64);
BQB_LAUNCH_DECL(128);
BQB_LAUNCH_DECL(160);
BQB_LAUNCH_DECL(256);
cudaError_t launch_score(const ScoreArgs &a, int n_inst, int sm_count, cudaStream_t stream, int *grid_x) {
    switch (a.lay.nsp_cap) {
        case 16: return launch_score_16(a, n_inst, sm_count, stream, grid_x);
        case 64: return launch_score_64(a, n_inst, sm_count, stream, grid_x);
        case 128: return launch_score_128(a, n_inst, sm_count, stream, grid_x);
        case 160: return launch_score_160(a, n_inst, sm_count, stream, grid_x);
        case 256: return launch_score_256(a, n_inst, sm_count, stream, grid_x);
        default: return cudaErrorInvalidValue;
    }
}
#elif defined(BQB_SCORE_REL)
#if BQB_SCORE_CLASS == 128
BQB_LAUNCH_REL_DECL(128) {
    if (smem_need<32, 1, 16, false, 512>(a, 0) <= SMEM_LIMIT)
        return launch_cfg<32, 1, 16, 1, false, 512, false, true, 24>(with_env(a), n_inst, sm_count, stream, grid_x);
    if (smem_need<32, 1, 16, true, 2048>(a, 2 * 32) <= SMEM_LIMIT)
        return launch_cfg<32, 1, 16, 1, true, 2048, false, true, 24>(with_env(a), n_inst, sm_count, stream, grid_x);
    return cudaErrorInvalidConfiguration;
}
#elif BQB_SCORE_CLASS == 160
BQB_LAUNCH_REL_DECL(160) {      // resident only up to ns = 128 here (the scratch of 16 warps), streamed above
    if (smem_need<40, 1, 16, false, 512>(a, 0) <= SMEM_LIMIT)
        return launch_cfg<40, 1, 16, 1, false, 512, false, true, 24>(with_env(a), n_inst, sm_count, stream, grid_x);
    if (smem_need<40, 1, 16, true, 2048>(a, 2 * 40) <= SMEM_LIMIT)
        return launch_cfg<40, 1, 16, 1, true, 2048, false, true, 24>(with_env(a), n_inst, sm_count, stream, grid_x);
    return cudaErrorInvalidConfiguration;
}
#elif BQB_SCORE_CLASS == 256
BQB_LAUNCH_REL_DECL(256) {      // (with >= 13 candidates the scratch rows of 16 warps leave no room for the chunk buffers)
    if (smem_need<64, 1, 16, true, 2048>(a, 2 * 64) <= SMEM_LIMIT)
        return launch_cfg<64, 1, 16, 1, true, 2048, false, true, 24>(with_env(a), n_inst, sm_count, stream, grid_x);
    return cudaErrorInvalidConfiguration;
}
#else
#error "band-relative kernels exist for the classes 128, 160 and 256"
#endif
#elif BQB_SCORE_CLASS == 16
BQB_LAUNCH_DECL(16) { return launch_cfg<4, 2, 8, 2, false, 2048, false, false>(a, n_inst, sm_count, stream, grid_x); }
#elif BQB_SCORE_CLASS == 64
// (rolled pairs, free-running warps and 4 x 4-warp CTAs were all slower with band skipping: 0.31 / 0.37 / 0.34 / 0.47 ms vs 0.28)
// (the band-relative loops <16, NT=1, 16 warps, BK=16> measured 0.364 ms against 0.286: at ns = 64 the band is most of the tile)
// Round-2 experiments on this class (profiles/score64_experiments_r02.md; 10^6 points, ns = 64, ms): this kernel 0.285; free
// running (ALIGN = 0) 0.335; barrier groups of 4 / 2 warps (ALIGN = 4 / 2) 0.284 / 0.293; rolled row-block loop 0.333; NT = 1
// with three CTAs per SM 0.43-0.57; 512-entry table 0.288; one CTA per SM 0.422 (=> T = 0.149 + 2.18 / warps: latency bound);
// a team kernel (cross-kernel tile shared by four warps through shared memory, 20-32 warps per SM) 0.298-0.333.
BQB_LAUNCH_DECL(64) { return launch_cfg<16, 2, 8, 2, false, 2048, 1, false>(a, n_inst, sm_count, stream, grid_x); }
#elif BQB_SCORE_CLASS == 128
BQB_LAUNCH_REL_DECL(128);
BQB_LAUNCH_DECL(128) {
    if (rel_variant() == 1) {
        const cudaError_t e = launch_score_rel_128(a, n_inst, sm_count, stream, grid_x);
        if (e != cudaErrorInvalidConfiguration) return e;
    }
    if (smem_need<32, 2, 8, false, 512>(a, 0) <= SMEM_LIMIT)
        return launch_cfg<32, 2, 8, 1, false, 512, false, true>(a, n_inst, sm_count, stream, grid_x);
    return launch_cfg<32, 2, 8, 1, true, 2048, false, true>(a, n_inst, sm_count, stream, grid_x);
}
#elif BQB_SCORE_CLASS == 160
BQB_LAUNCH_REL_DECL(160);
BQB_LAUNCH_DECL(160) {       // absolute tile: resident while the instances' operands fit (ns <= 136 ... 144 depending on the candidates), then streamed
    if (rel_variant() == 1) {
        const cudaError_t e = launch_score_rel_160(a, n_inst, sm_count, stream, grid_x);
        if (e != cudaErrorInvalidConfiguration) return e;
    }
    if (smem_need<40, 2, 8, false, 512>(a, 0) <= SMEM_LIMIT)
        return launch_cfg<40, 2, 8, 1, false, 512, false, true>(a, n_inst, sm_count, stream, grid_x);
    return launch_cfg<40, 2, 8, 1, true, 2048, false, true>(a, n_inst, sm_count, stream, grid_x);
}
#elif BQB_SCORE_CLASS == 256
BQB_LAUNCH_REL_DECL(256);
BQB_LAUNCH_DECL(256) {
    if (rel_variant() == 1) {
        const cudaError_t e = launch_score_rel_256(a, n_inst, sm_count, stream, grid_x);
        if (e != cudaErrorInvalidConfiguration) return e;
    }
    return launch_cfg<64, 1, 8, 1, true, 2048, false, true>(a, n_inst, sm_count, stream, grid_x);
}
#else
#error "BQB_SCORE_CLASS must be 16, 64, 128, 160 or 256"
#endif

}  // namespace bqb
