// Setup kernel: one CTA per model instance (one BQ problem under one hyper-parameter set) with the working matrix
// RESIDENT IN SHARED MEMORY as a packed lower triangle (row i starts at i (i + 1) / 2).
//
// It replaces, once per instance instead of once per query point, what the reference does through the `gp` package
// and linalg_c (Gram build bq.py:465, dpotrf linalg_c.pyx:86, gp.mean / cov bq.py:493-496), computes Z_mean
// (bq_c.pyx:157-213), Z_var (bq_c.pyx:264-355 with gauss_c.pyx:416-531 / :235-339 fused) and log_lh (bq.py:546),
// and emits the operands of the scoring kernel in DMMA fragment order.
//
// Why it is built this way (an earlier kernel with dense matrices in global scratch, profiles/ncu_setup_r01: FP64 pipe
// 10 % busy, 57 % of the stall samples on CTA barriers behind one-warp / one-thread phases, 440 MB of global scratch
// thrashing the L2 at C5 scale):
//   * ONE packed triangle serves K_tl -> L_tl -> L_tl^-1 (in place), then K_l -> L -> [L_ss^-1; C L_cc] (in place),
//     then (s_l != 0 only) K_l + s_l^2 I.  n (n + 1) / 2 doubles: 92 KB at n = 152.  Two CTAs of 256 threads per SM
//     while two instances fit (n <= 155 with ten candidates; decided by the occupancy query at launch) and the launch
//     fills the SMs more than once, one CTA of 512 threads up to n = 218; larger instances (the 256 and 512 classes)
//     run the same code on a packed triangle in global scratch.
//   * Cholesky by panels of 8: the 8 x 8 diagonal block is factorised by eight lanes in registers (shuffles; rsqrt with
//     one Newton step instead of sqrt + divide), the panel below is a column-oriented forward substitution with one
//     thread per row, the trailing update is DMMA (two mma.m8n8k4 per 8 x 8 block).  Three barriers per panel.
//   * Triangular inverse in place by block rows of 8: the block row of L is staged, a warp per block column J
//     accumulates R = sum_K L_IK X_KJ by DMMA and solves L_II X_IJ = -R inside its accumulator fragment (rows exchanged
//     by shuffles).  Every column of the result is a forward substitution L x = e_c, i.e. backward stable column by
//     column; multiplying by explicit inverses of the 8 x 8 diagonal blocks instead was 37x less accurate at
//     cond(K_tl) = 3.5e9 (tests/golden/illcond_b).
//   * The candidates' guard (bq.py:942-947) evaluates the cross-kernel once per candidate instead of once per row, four
//     candidates per pass; the symmetric n x n integral matrix of Z_var is evaluated for i <= j only; the inner loops of
//     Z_var multiply by reciprocals instead of dividing; L_tl^-1 is read back from its fragment-ordered copy in the
//     model block for beta' K_tl^-1 beta.
#include <cstdio>

#include "bq_common.cuh"

namespace bqb {

constexpr int S2_NVEC_FIXED = 5;     // tl_s, a_tl, x_sc, l_sc, rdiag: live across the triangular inverses
constexpr int S2_NVEC_UNION = 9;     // b_sc, u_s, ua_s, gg, ga, alpha, beta, tmp, tmp2: share their space with the stage
constexpr double S2_LOG_2PI = 1.8378770664093453;
constexpr double S2_SQRT_2PI = 2.5066282746310002;

__host__ __device__ __forceinline__ int tri(int i) { return (i * (i + 1)) >> 1; }

// shared-memory carve-up (doubles) for instances of order <= nmax with <= ncm candidates
struct S2Carve {
    int np, lds, nv, un, small, total;
};
__host__ __device__ inline S2Carve s2_carve(int nmax, int ncm, bool tsmem) {
    S2Carve c;
    c.np = tsmem ? ((tri(nmax) + 1) & ~1) : 0;
    c.lds = (((nmax + 7) & ~7) + 1) | 1;            // a staged block row reaches column round8(n) - 1; odd stride
    c.nv = (nmax + 1) & ~1;
    const int a = 8 * c.lds, b = S2_NVEC_UNION * c.nv;
    c.un = ((a > b ? a : b) + 1) & ~1;
    c.small = 2 * ncm * ncm + 2;
    c.total = c.np + S2_NVEC_FIXED * c.nv + c.un + 144 + c.small;
    return c;
}

// e = tri(i) + j with 0 <= j <= i
__device__ __forceinline__ void tri_decode(int e, int &i, int &j) {
    int r = (int)((sqrtf(8.0f * (float)e + 1.0f) - 1.0f) * 0.5f);
    if (tri(r + 1) <= e) ++r;
    else if (tri(r) > e) --r;
    i = r;
    j = e - tri(r);
}

// Tolerance of np.isclose(x_a, x_s, atol=1e-4) (bq.py:456): atol + rtol |x_s| rounded after the product and after the
// sum, as numpy evaluates it.  Contracted to one fma it differs by an ulp for about a fifth of all x_s, and a point at
// that distance would take the shortcut where the reference does not (or the other way round).
__device__ __forceinline__ double isclose_tol(double xs) { return __dadd_rn(1e-4, __dmul_rn(1e-5, fabs(xs))); }

template <int NT>
__device__ double block_sum2(double v, double *red) {
    v = warp_sum(v);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) red[w] = v;
    __syncthreads();
    double s = 0;
#pragma unroll
    for (int i = 0; i < NT / 32; ++i) s += red[i];   // fixed order: deterministic
    return s;
}

template <int NT>
__device__ double block_max2(double v, double *red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) red[w] = v;
    __syncthreads();
    double s = red[0];
#pragma unroll
    for (int i = 1; i < NT / 32; ++i) s = fmax(s, red[i]);
    return s;
}

#ifdef BQB_SETUP_PROF
__device__ long long g_s2_sub[8];
#define SUBT(i, t0) do { if (threadIdx.x == 0 && blockIdx.x == 0) g_s2_sub[i] += clock64() - (t0); } while (0)
#define SUBT0() clock64()
#else
#define SUBT(i, t0) do { } while (0)
#define SUBT0() 0
#endif

// Factorises the 8 x 8 diagonal block at jb (w = min(8, n - jb) live rows) with eight lanes of the calling warp: lane r
// holds row r in registers, columns are exchanged by shuffles.  Writes the block back to T, its rows to Lb[8][8], the
// reciprocals of its diagonal to Rb[8] and rdiag[jb ..]; a non-positive pivot j sets *s_info = jb + j + 1.
__device__ __forceinline__ void chol_diag_block(double *T, int n, int jb, double *Lb, double *Rb, double *rdiag, int *s_info) {
    const int lane = threadIdx.x & 31;
    const int w = (n - jb < 8) ? n - jb : 8;
    double d[8], rsv[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        double v = (c == lane) ? 1.0 : 0.0;                        // identity rows past the matrix edge
        if (lane < w && c <= lane) v = T[tri(jb + lane) + jb + c];
        d[c] = v;
    }
    int info = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const double piv = __shfl_sync(0xffffffffu, d[j], j);
        if (!(piv > 0.0) && info == 0) info = jb + j + 1;          // warp uniform
        // l = sqrt(piv), rs = 1 / l: rsqrt refined by one Newton step each (an unrefined rsqrt, 1 ulp and not
        // unbiased, cost a factor 10 of accuracy at cond 3.5e9)
        double rs = rsqrt(piv);
        double l = piv * rs;
        l = fma(0.5 * rs, fma(-l, l, piv), l);
        rs = fma(rs, fma(-l, rs, 1.0), rs);
        rsv[j] = rs;
        if (lane == j) d[j] = l;
        else if (lane > j) d[j] *= rs;
#pragma unroll
        for (int k = j + 1; k < 8; ++k) {
            const double lkj = __shfl_sync(0xffffffffu, d[j], k);
            if (lane >= k) d[k] = fma(-d[j], lkj, d[k]);      // (a separate lane == k case without the shuffle: 2.8x slower, branches)
        }
    }
    if (lane < 8) {
#pragma unroll
        for (int c = 0; c < 8; ++c) Lb[lane * 8 + c] = d[c];
        if (lane == 0) {
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                Rb[c] = rsv[c];
                if (c < w) rdiag[jb + c] = rsv[c];
            }
        }
    }
    if (info == 0 && lane < w) {
#pragma unroll
        for (int c = 0; c < 8; ++c)
            if (c <= lane) T[tri(jb + lane) + jb + c] = d[c];
    }
    if (lane == 0 && info) *s_info = info;
}

// One 8 x 8 block of the trailing update: T[i0 + r][k0 + c] -= P[i0 + r] . P[k0 + c], P = columns jb .. jb + 7.
// a0 / a1: this lane's (negated) A fragments of the row block; rowa = tri(i0 + lr); va = i0 + lr < n.
__device__ __forceinline__ void chol_trail_block(double *T, int n, int jb, int k0, int ia, int rowa, bool va, double a0, double a1) {
    const int lane = threadIdx.x & 31, lr = lane >> 2, lc = lane & 3;
    const int rb = k0 + lr;
    double b0 = 0.0, b1 = 0.0;
    if (rb < n) { const double *p = T + tri(rb) + jb + lc; b0 = p[0]; b1 = p[4]; }
    const int cc = k0 + 2 * lc;
    double *pc = T + rowa + cc;
    const bool v0 = va && (cc <= ia), v1 = va && (cc + 1 <= ia);
    double c0 = v0 ? pc[0] : 0.0, c1 = v1 ? pc[1] : 0.0;
    dmma(c0, c1, a0, b0);
    dmma(c0, c1, a1, b1);
    if (v0) pc[0] = c0;
    if (v1) pc[1] = c1;
}

// In-place lower Cholesky of the packed n x n matrix T.  Returns 0, or j + 1 when pivot j is not positive (LAPACK
// dpotrf's info, linalg_c.pyx:86-91).  rdiag[j] <- 1 / L[j][j].  blk: 2 x 72 doubles of shared scratch (the factorised
// diagonal block and the reciprocals of its diagonal, double buffered).
// Right-looking by panels of 8 with one panel of look-ahead: after the panel solve, all warps update the FIRST block column
// of the trailing matrix; then warp 0 factorises the next diagonal block (a chain of eight dependent rsqrt steps, ~2.4 k
// cycles) while the other warps update the remaining block columns, each warp walking a contiguous run of blocks row by
// row (A fragments reloaded only on a row change, addresses advanced incrementally: the first version spent ~190
// instructions per two DMMAs on index arithmetic and was issue bound).
template <int NT>
__device__ int chol_packed(double *T, int n, double *blk, int *s_info, double *rdiag) {
    constexpr int NW = NT / 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int lr = lane >> 2, lc = lane & 3;
    if (tid == 0) *s_info = 0;
    __syncthreads();
    long long tp = SUBT0();
    if (warp == 0) chol_diag_block(T, n, 0, blk, blk + 64, rdiag, s_info);
    __syncthreads();
    SUBT(0, tp);
    int pb = 0;
    for (int jb = 0; jb < n; jb += 8, pb ^= 1) {
        if (*s_info) return *s_info;
        const double *Lb = blk + pb * 72, *Rb = Lb + 64;
        const int t0 = jb + 8;
        const int nbelow = n - t0;
        if (nbelow <= 0) break;
        tp = SUBT0();
        // panel: P_i L_D^T = A_i[jb : jb + 8] for the rows below the block: forward substitution, one thread per row
        // (column oriented: after p_c is known the remaining right-hand sides are updated by independent FMAs).  A
        // multiplication by the explicit inverse of the block would be cheaper but is not backward stable, and the
        // 8 x 8 blocks of a smooth kernel matrix are badly conditioned themselves.
        for (int i = tid; i < nbelow; i += NT) {
            double *row = T + tri(t0 + i) + jb;
            double sv[8];
#pragma unroll
            for (int c = 0; c < 8; ++c) sv[c] = row[c];
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const double pc = sv[c] * Rb[c];
                sv[c] = pc;
#pragma unroll
                for (int k = c + 1; k < 8; ++k) sv[k] = fma(-pc, Lb[k * 8 + c], sv[k]);
            }
#pragma unroll
            for (int c = 0; c < 8; ++c) row[c] = sv[c];
        }
        __syncthreads();
        SUBT(1, tp);
        tp = SUBT0();
        const int m = (nbelow + 7) >> 3;
        // first block column of the trailing matrix (it holds the next diagonal block and the next panel)
        for (int bi = warp; bi < m; bi += NW) {
            const int ia = t0 + 8 * bi + lr;
            const bool va = ia < n;
            double a0 = 0.0, a1 = 0.0;
            if (va) { const double *p = T + tri(ia) + jb + lc; a0 = -p[0]; a1 = -p[4]; }
            chol_trail_block(T, n, jb, t0, ia, tri(ia), va, a0, a1);
        }
        __syncthreads();
        SUBT(2, tp);
        tp = SUBT0();
        if (warp == 0) {
            chol_diag_block(T, n, t0, blk + (pb ^ 1) * 72, blk + (pb ^ 1) * 72 + 64, rdiag, s_info);
        } else if (m > 1) {
            // blocks (bi, bk) with 1 <= bk <= bi < m, flattened row by row: g = tri(bi - 1) + (bk - 1)
            const int total = tri(m - 1);
            const int q = (total + NW - 2) / (NW - 1);
            int g = (warp - 1) * q;
            const int gend = (g + q < total) ? g + q : total;
            if (g < gend) {
                int bi, bk;
                tri_decode(g, bi, bk);
                bi += 1; bk += 1;
                while (g < gend) {
                    const int ia = t0 + 8 * bi + lr;
                    const bool va = ia < n;
                    const int rowa = tri(ia);
                    double a0 = 0.0, a1 = 0.0;
                    if (va) { const double *p = T + rowa + jb + lc; a0 = -p[0]; a1 = -p[4]; }
                    for (; bk <= bi && g < gend; ++bk, ++g) chol_trail_block(T, n, jb, t0 + 8 * bk, ia, rowa, va, a0, a1);
                    bi += 1; bk = 1;
                }
            }
        }
        __syncthreads();
        SUBT(5, tp);
    }
    return *s_info;
}

// T[0:n, 0:n] <- its inverse (lower triangular, packed, in place); rows >= n of T are not touched.  Block forward
// substitution by block rows of 8 (see the header comment).  rdiag: reciprocals of L's diagonal (from chol_packed).
// stage: 8 x lds doubles of shared scratch.
template <int NT>
__device__ void tri_inverse_packed(double *T, int n, double *stage, int lds, const double *rdiag) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int lr = lane >> 2, lc = lane & 3;
    for (int ib = 0; ib < n; ib += 8) {
        const int h = (n - ib < 8) ? n - ib : 8;
        long long tp = SUBT0();
        const int wd = ib + 8;
        for (int e = tid; e < 8 * wd; e += NT) {
            const int r = e / wd, k = e - r * wd;
            double v = 0.0;
            if (r < h && k <= ib + r) v = T[tri(ib + r) + k];
            stage[r * lds + k] = v;
        }
        __syncthreads();
        SUBT(3, tp);
        tp = SUBT0();
        const int nJ = ib >> 3;
        for (int J = warp; J <= nJ; J += NT / 32) {
            double c0 = 0.0, c1 = 0.0, e0 = 0.0, e1 = 0.0;
            const int jc = 8 * J + lr;
            if (8 * J < ib) {
                // operands of K-step K + 1 are loaded before the DMMAs of K-step K; only K = J touches the diagonal
                // block of X (its upper part reads as zero)
                int kb = 8 * J;
                const double *sa = stage + lr * lds + lc;
                double a0 = sa[kb], a1 = sa[kb + 4];
                double b0 = (jc <= kb + lc) ? T[tri(kb + lc) + jc] : 0.0;
                double b1 = (jc <= kb + 4 + lc) ? T[tri(kb + 4 + lc) + jc] : 0.0;
                for (kb += 8; kb < ib; kb += 8) {
                    const double a0n = sa[kb], a1n = sa[kb + 4];
                    const double b0n = T[tri(kb + lc) + jc], b1n = T[tri(kb + 4 + lc) + jc];
                    dmma(c0, c1, a0, b0);
                    dmma(e0, e1, a1, b1);
                    a0 = a0n; a1 = a1n; b0 = b0n; b1 = b1n;
                }
                dmma(c0, c1, a0, b0);
                dmma(e0, e1, a1, b1);
            }
            double x0 = -(c0 + e0), x1 = -(c1 + e1);
            if (J == nJ) { x0 = (lr == 2 * lc) ? 1.0 : 0.0; x1 = (lr == 2 * lc + 1) ? 1.0 : 0.0; }
            const double *Lrow = stage + lr * lds + ib;                  // row lr of L_II
            const double rinv = (lr < h) ? rdiag[ib + lr] : 1.0;
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                if (lr == r) { x0 *= rinv; x1 *= rinv; }
                const double xr0 = __shfl_sync(0xffffffffu, x0, r * 4 + lc), xr1 = __shfl_sync(0xffffffffu, x1, r * 4 + lc);
                if (lr > r) {
                    const double l = Lrow[r];
                    x0 = fma(-l, xr0, x0);
                    x1 = fma(-l, xr1, x1);
                }
            }
            if (lr < h) {
                double *p = T + tri(ib + lr) + 8 * J + 2 * lc;
                if (J < nJ) { p[0] = x0; p[1] = x1; }
                else {
                    if (2 * lc <= lr) p[0] = x0;
                    if (2 * lc + 1 <= lr) p[1] = x1;
                }
            }
        }
        __syncthreads();
        SUBT(4, tp);
    }
}

// o1[i] = sum_{k <= i} X[i][k] v1[k] (and the same for v2 -> o2 when v2 is given); warp per row
template <int NT>
__device__ void lower_matvec_p(const double *T, int n, const double *v1, double *o1, const double *v2, double *o2) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = warp; i < n; i += NT / 32) {
        const double *row = T + tri(i);
        double s1 = 0.0, s2 = 0.0;
        for (int k = lane; k <= i; k += 32) {
            const double x = row[k];
            s1 = fma(x, v1[k], s1);
            if (v2) s2 = fma(x, v2[k], s2);
        }
        s1 = warp_sum(s1);
        if (v2) s2 = warp_sum(s2);
        if (lane == 0) {
            o1[i] = s1;
            if (v2) o2[i] = s2;
        }
    }
    __syncthreads();
}

// o1[c] = sum_{i >= c} X[i][c] v1[i], the same for v2 -> o2 when given; one thread per column
// (NT = 512 and n <= 256: both right-hand sides at once, threads 0 .. 255 and 256 .. 511)
template <int NT>
__device__ void lower_matvec_t_p(const double *T, int n, const double *v1, double *o1, const double *v2, double *o2) {
    const bool split = NT == 512 && n <= 256;
    const int cols = split ? 256 : NT;
    for (int h0 = 0; h0 < 2; h0 += split ? 2 : 1) {
        const int half = split ? (int)(threadIdx.x >> 8) : h0;
        const double *v = half ? v2 : v1;
        double *o = half ? o2 : o1;
        if (v == nullptr) continue;
        for (int c = split ? (int)(threadIdx.x & 255) : (int)threadIdx.x; c < n; c += cols) {
            double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
            int i = c;
            for (; i + 3 < n; i += 4) {
                s0 = fma(T[tri(i) + c], v[i], s0);
                s1 = fma(T[tri(i + 1) + c], v[i + 1], s1);
                s2 = fma(T[tri(i + 2) + c], v[i + 2], s2);
                s3 = fma(T[tri(i + 3) + c], v[i + 3], s3);
            }
            for (; i < n; ++i) s0 = fma(T[tri(i) + c], v[i], s0);
            o[c] = (s0 + s1) + (s2 + s3);
        }
    }
    __syncthreads();
}

// dst <- the fragment-ordered copy of c * X (triangular operand of the scoring kernel), zeros in the padding
template <int NT>
__device__ void write_tri_frags(const double *T, int ns, double c, double *dst, int nb_cap) {
    const int total = tri_frags(nb_cap) * 32;
    for (int e = threadIdx.x; e < total; e += NT) {
        const int f = e >> 5, l = e & 31;
        int rb = (int)((sqrtf(4.0f * (float)f + 1.0f) - 1.0f) * 0.5f);      // largest rb with rb (rb + 1) <= f
        if ((rb + 1) * (rb + 2) <= f) ++rb;
        else if (rb * (rb + 1) > f) --rb;
        const int ks = f - rb * (rb + 1);
        const int r = 8 * rb + (l >> 2), k = 4 * ks + (l & 3);
        dst[e] = (r < ns && k <= r) ? c * T[tri(r) + k] : 0.0;
    }
}

// gauss_c.pyx:20-62 for d = 1 with L = sqrt(var), logdet = 2 log L
__device__ __forceinline__ double mvn_logpdf1b(double x, double m, double L, double logdet) {
    const double diff = x - m;
    const double buf = (diff / L) / L;
    return -0.5 * ((S2_LOG_2PI + logdet) + diff * buf);
}
// the same with rL = 1 / L (inner loops)
__device__ __forceinline__ double mvn_logpdf1r(double x, double m, double rL, double logdet) {
    const double diff = x - m;
    const double buf = (diff * rL) * rL;
    return -0.5 * ((S2_LOG_2PI + logdet) + diff * buf);
}

// -DBQB_SETUP_PROF: CTA 0 prints the clock64() count of every phase (bench_micro/setup_prof2.py)
#ifdef BQB_SETUP_PROF
#define PH(i) do { __syncthreads(); if (threadIdx.x == 0 && blockIdx.x == 0) s_prof[i] = clock64(); } while (0)
#else
#define PH(i) do { } while (0)
#endif

template <bool TSMEM, int NT, int KIND>
__global__ void __launch_bounds__(NT, 512 / NT) bq_setup2_kernel(SetupArgs a) {
#ifdef BQB_SETUP_PROF
    __shared__ long long s_prof[24];
    if (threadIdx.x == 0 && blockIdx.x == 0)
        for (int i = 0; i < 8; ++i) g_s2_sub[i] = 0;
#endif
    constexpr int NW = NT / 32;
    __shared__ double red[NW];
    __shared__ int s_fail, s_info;
    extern __shared__ double s_dyn[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int inst = a.inst_list ? a.inst_list[a.inst0 + blockIdx.x] : a.inst0 + blockIdx.x;
    const int ns = a.ns[inst], nc = a.nc[inst], n = ns + nc;
    const Layout &lay = a.lay;
    double *M = a.models + (size_t)inst * lay.total;

    // shared-memory carve-up: [T packed] [5 vectors] [9 vectors | stage 8 x lds] [blk 2 x 72] [Kcc, S0]
    const int nmax = a.n_max, ncm = a.nc_max;
    const S2Carve cv = s2_carve(nmax, ncm, TSMEM);
    const int lds = cv.lds, nv = cv.nv;
    double *T = TSMEM ? s_dyn : a.work + (size_t)blockIdx.x * a.work_stride;
    double *vec = s_dyn + cv.np;
    double *tl_s = vec, *a_tl = vec + nv, *x_sc = vec + 2 * nv, *l_sc = vec + 3 * nv, *rdiag = vec + 4 * nv;
    double *un = vec + S2_NVEC_FIXED * nv;
    double *stage = un;
    double *b_sc = un, *u_s = un + nv, *ua_s = un + 2 * nv, *gg = un + 3 * nv, *ga = un + 4 * nv, *alpha = un + 5 * nv,
           *beta = un + 6 * nv, *tmp = un + 7 * nv, *tmp2 = un + 8 * nv;
    double *blk = un + cv.un;
    double *Kcc = blk + 144;                      // ncm^2, kept for the Schur complement
    double *S0 = Kcc + ncm * ncm;                 // ncm^2

    // header, vectors and the dense operand rows are zeroed (padding must be exact zeros); the triangular operand
    // arrays are written in full by write_tri_frags
    PH(0);
    for (int i = tid; i < lay.n_small; i += NT) M[i] = 0.0;
    for (int i = tid; i < 3 * lay.nks_cap * 32; i += NT) M[lay.off_af_l_dense + i] = 0.0;
    if (tid == 0) s_fail = SETUP_OK;
    __syncthreads();

    const double h_tl = a.hyp[inst * 6 + 0], w_tl = a.hyp[inst * 6 + 1], s_tl = a.hyp[inst * 6 + 2];
    const double h_l = a.hyp[inst * 6 + 3], w_l = a.hyp[inst * 6 + 4], s_l = a.hyp[inst * 6 + 5];
    const double mu = a.prior[inst * 3 + 0], sig2 = a.prior[inst * 3 + 1], thresh = a.prior[inst * 3 + 2];

    // ---- P0 validate (sizes first: everything below indexes shared memory with them)
    if (!(ns >= 1 && ns <= lay.nsp_cap && nc >= 0 && nc <= NC_MAX && nc <= ncm && n <= nmax)) {
        if (tid == 0) M[H_STATUS] = SETUP_BAD_INPUT;
        return;
    }
    {
        const double *x_s = a.x_s + (size_t)inst * a.in_stride;
        const double *l_s = a.l_s + (size_t)inst * a.in_stride;
        const double *x_c = a.x_c + (size_t)inst * NC_MAX;
        int bad = 0;
        for (int i = tid; i < ns; i += NT) {
            const double x = x_s[i], l = l_s[i];
            bad |= !(isfinite(x) && isfinite(l) && l > 0.0);
            tmp[i] = x;
            tmp2[i] = l;
        }
        for (int i = tid; i < nc; i += NT) {
            const double x = x_c[i];
            bad |= !isfinite(x);
            x_sc[ns + i] = x;
        }
        if (tid == 0) {
            bad |= !(h_tl > 0 && w_tl > 0 && s_tl >= 0 && h_l > 0 && w_l > 0 && s_l >= 0 && sig2 > 0 && isfinite(mu));
            if (KIND) bad |= !(a.period && a.period[inst * 2] > 0 && a.period[inst * 2 + 1] > 0);
        }
        if (bad) s_fail = SETUP_BAD_INPUT;
    }
    __syncthreads();
    if (s_fail) { if (tid == 0) M[H_STATUS] = s_fail; return; }

    // ---- P0b: observations in ascending order of x (stable rank sort).  Every result of this kernel and of the scoring
    // kernel is invariant under a permutation of the observations (up to rounding), and with sorted observations the
    // k-steps that matter for a query point are few and contiguous (band skipping, bq_score.cu) whatever order the
    // caller -- or add_observation, which appends -- left them in.  Already sorted input is left exactly as it is.
    for (int i = tid; i < ns; i += NT) {
        const double xi = tmp[i];
        int rank = 0;
        for (int j = 0; j < ns; ++j) {
            const double xj = tmp[j];
            rank += (xj < xi) || (xj == xi && j < i);
        }
        x_sc[rank] = xi;
        l_sc[rank] = tmp2[i];
    }
    __syncthreads();

    PH(1);
    // kernel = c exp(nh D^2): gp.GaussianKernel (D = d, c = h^2 / (sqrt(2 pi) w)) or gp.PeriodicKernel (D = 2 sin(d / 2p), c = h^2)
    constexpr int kind = KIND;                          // (a template parameter: the Gaussian instantiation carries no sin code)
    const double hp_tl = kind ? 0.5 / a.period[inst * 2] : 0.0, hp_l = kind ? 0.5 / a.period[inst * 2 + 1] : 0.0;
    const double c_tl = kind ? h_tl * h_tl : (h_tl * h_tl) / (S2_SQRT_2PI * w_tl), nh_tl = -0.5 / (w_tl * w_tl);
    const double c_l = kind ? h_l * h_l : (h_l * h_l) / (S2_SQRT_2PI * w_l), nh_l = -0.5 / (w_l * w_l);
    // trapezoid approximation of the integrals over a grid xo (bq_c.pyx:216-261, :358-422, :538-598) instead of the
    // closed forms: wp[j] = (trapezoid weight of xo[j]) x (prior density at xo[j])
    const int n_xo = a.n_xo;
    const double *xo = n_xo ? a.xo + (size_t)inst * a.xo_stride : nullptr;
    double *wp = n_xo ? a.wp + (size_t)inst * n_xo : nullptr;
    double *gz = n_xo ? a.gz + (size_t)blockIdx.x * n_xo : nullptr;
    if (n_xo) {
        const double *pxo = a.pxo + (size_t)inst * a.xo_stride;
        for (int j = tid; j < n_xo; j += NT) {
            const double tw = 0.5 * ((j > 0 ? xo[j] - xo[j - 1] : 0.0) + (j + 1 < n_xo ? xo[j + 1] - xo[j] : 0.0));
            wp[j] = tw * pxo[j];
        }
    }

    // ---- P1/P2: tl_s = log l_s (bq.py:73); K_tl = K(x_s, x_s) + s_tl^2 I, lower triangle
    for (int i = tid; i < ns; i += NT) tl_s[i] = log(l_sc[i]);
    for (int e = tid; e < tri(ns); e += NT) {
        int i, j;
        tri_decode(e, i, j);
        double v = c_tl * kernel_exp(x_sc[i] - x_sc[j], nh_tl, kind, hp_tl);
        if (i == j) v += s_tl * s_tl;
        T[e] = v;
    }
    __syncthreads();
    PH(2);
    // ---- P3: L_tl
    if (chol_packed<NT>(T, ns, blk, &s_info, rdiag)) { if (tid == 0) M[H_STATUS] = SETUP_KTL_NOTPD; return; }
    PH(3);
    double sumlog_tl;
    {
        double p = 0.0;
        for (int i = tid; i < ns; i += NT) p += log(T[tri(i) + i]);
        sumlog_tl = block_sum2<NT>(p, red);
    }
    PH(4);
    // ---- P4: L_tl^-1 in place, and its fragment-ordered copy
    tri_inverse_packed<NT>(T, ns, stage, lds, rdiag);
    PH(5);
    write_tri_frags<NT>(T, ns, c_tl, M + lay.off_af_tl_tri, lay.nb_cap);
    PH(6);
    // ---- P5: a_tl = K_tl^-1 tl_s
    lower_matvec_p<NT>(T, ns, tl_s, tmp, nullptr, nullptr);
    lower_matvec_t_p<NT>(T, ns, tmp, a_tl, nullptr, nullptr);
    PH(7);
    // ---- P6: l_c = exp(gp_log_l.mean(x_c))  (bq.py:985 / :942-950), four candidates per pass:
    //      stage rows 0..3 = K_tl(x_c[j], x_s), rows 4..7 = (L_tl^-1 k_j)^2 element-wise (the guard only)
    for (int j0 = 0; j0 < nc; j0 += 4) {
        const int nbt = (nc - j0 < 4) ? nc - j0 : 4;
        for (int e = tid; e < nbt * ns; e += NT) {
            const int j = e / ns, k = e - j * ns;
            stage[j * lds + k] = c_tl * kernel_exp(x_sc[ns + j0 + j] - x_sc[k], nh_tl, kind, hp_tl);
        }
        __syncthreads();
        if (a.check_max) {
            for (int e = tid; e < nbt * ns; e += NT) {
                const int j = e / ns, r = e - j * ns;
                const double *row = T + tri(r), *kc = stage + j * lds;
                double s0 = 0.0, s1 = 0.0;
                int k = 0;
                for (; k + 1 <= r; k += 2) {
                    s0 = fma(row[k], kc[k], s0);
                    s1 = fma(row[k + 1], kc[k + 1], s1);
                }
                if (k <= r) s0 = fma(row[k], kc[k], s0);
                const double y = s0 + s1;
                stage[(4 + j) * lds + r] = y * y;
            }
            __syncthreads();
        }
        if (warp < nbt) {
            const int j = warp;
            double m = 0.0, q = 0.0;
            for (int k = lane; k < ns; k += 32) {
                m = fma(stage[j * lds + k], a_tl[k], m);
                if (a.check_max) q += stage[(4 + j) * lds + k];
            }
            m = warp_sum(m);
            q = warp_sum(q);
            if (lane == 0) {
                if (a.check_max) {
                    // V = diag(cov(x_c)) = ktt - |L_tl^-1 k|^2 ; LinAlgError if m + 2 sqrt(max(V, 0)) > MAX
                    double V = c_tl - q;
                    if (V < 0) V = 0;
                    if (m + 2 * sqrt(V) > MAX_EXPONENT) s_fail = SETUP_MEAN_TOO_LARGE;
                }
                const double lc = exp(m);
                M[lay.off_lc + j0 + j] = lc;
                l_sc[ns + j0 + j] = lc;
            }
        }
        __syncthreads();
    }
    __syncthreads();
    if (s_fail) { if (tid == 0) M[H_STATUS] = s_fail; return; }

    PH(8);
    // ---- P7: K_l(x_sc, x_sc) without s_l^2 (the bordered matrix of bq.py:465 is Kxoxo) -> L
    for (int e = tid; e < tri(n); e += NT) {
        int i, j;
        tri_decode(e, i, j);
        T[e] = c_l * kernel_exp(x_sc[i] - x_sc[j], nh_l, kind, hp_l);
    }
    __syncthreads();
    PH(9);
    for (int e = tid; e < nc * nc; e += NT) {
        const int i = e / nc, j = e - i * nc;
        const int hi = i > j ? i : j, lo = i > j ? j : i;
        Kcc[i * ncm + j] = T[tri(ns + hi) + ns + lo];
    }
    if (chol_packed<NT>(T, n, blk, &s_info, rdiag)) { if (tid == 0) M[H_STATUS] = SETUP_KL_NOTPD; return; }
    PH(10);
    double sumlog_l;
    {
        double p = 0.0;
        for (int i = tid; i < n; i += NT) p += log(T[tri(i) + i]);
        sumlog_l = block_sum2<NT>(p, red);
    }
    PH(11);
    // ---- P8: L_ss^-1 in place (rows ns .. n - 1 keep [C L_cc])
    tri_inverse_packed<NT>(T, ns, stage, lds, rdiag);
    PH(12);
    // ---- P9: b_sc = int_K (gauss_c.pyx:95-164): h^2 exp(mvn_logpdf(x; mu, w_l^2 + sigma2))
    const double var_b = sig2 + w_l * w_l;
    const double Lb = sqrt(var_b), logdet_b = 2 * log(Lb);
    if (n_xo) {
        // int_K by the trapezoid rule (bq_c.pyx:585-593): sum_j wp[j] K_l(x_i, xo[j]), a warp per row
        __syncthreads();                                 // wp is complete
        for (int i = warp; i < n; i += NW) {
            const double xi = x_sc[i];
            double sacc = 0.0;
            for (int j = lane; j < n_xo; j += 32) sacc = fma(wp[j], kernel_exp(xi - xo[j], nh_l, kind, hp_l), sacc);
            sacc = warp_sum(sacc);
            if (lane == 0) b_sc[i] = c_l * sacc;
        }
    } else {
        for (int i = tid; i < n; i += NT) b_sc[i] = (h_l * h_l) * exp(mvn_logpdf1b(x_sc[i], mu, Lb, logdet_b));
    }
    __syncthreads();
    PH(13);
    // ---- P10: pattern-independent pieces
    lower_matvec_p<NT>(T, ns, b_sc, u_s, l_sc, ua_s);       // u_s = L_ss^-1 b_s ; ua_s = L_ss^-1 l_s
    lower_matvec_t_p<NT>(T, ns, u_s, gg, ua_s, ga);         // g_gamma = L_ss^-T u_s ; g_alpha = L_ss^-T ua_s
    PH(14);
    const int nsp = (ns + 7) & ~7, nks = nsp / 4;
    const int ndb = (nc + 2 + 7) / 8;
    // dense operand rows: c_l W (W[j][k] = -sum_{i >= k} C[j][i] Linv[i][k], C = L[ns + j][0:ns]), c_l g_gamma, c_l g_alpha
    for (int e = tid; e < (nc + 2) * ns; e += NT) {
        const int r = e / ns, k = e - r * ns;
        double v;
        if (r < nc) {
            const double *C = T + tri(ns + r);
            double s0 = 0.0, s1 = 0.0;
            int i = k;
            for (; i + 1 < ns; i += 2) {
                s0 = fma(C[i], T[tri(i) + k], s0);
                s1 = fma(C[i + 1], T[tri(i + 1) + k], s1);
            }
            if (i < ns) s0 = fma(C[i], T[tri(i) + k], s0);
            v = c_l * -(s0 + s1);
        } else {
            v = c_l * (r == nc ? gg[k] : ga[k]);
        }
        M[lay.off_af_l_dense + (((r >> 3) * nks + (k >> 2)) << 5) + ((r & 7) << 2) + (k & 3)] = v;
    }
    PH(15);
    // wb = b_c - C u_s ; wa = l_c - C ua_s ; S0 = K_cc - C C^T  (warp per output)
    for (int j = warp; j < nc; j += NW) {
        const double *C = T + tri(ns + j);
        double s1 = 0.0, s2 = 0.0;
        for (int i = lane; i < ns; i += 32) {
            const double c = C[i];
            s1 = fma(c, u_s[i], s1);
            s2 = fma(c, ua_s[i], s2);
        }
        s1 = warp_sum(s1);
        s2 = warp_sum(s2);
        if (lane == 0) { M[lay.off_wb + j] = b_sc[ns + j] - s1; M[lay.off_wa + j] = l_sc[ns + j] - s2; }
    }
    for (int e = warp; e < nc * nc; e += NW) {
        const int i = e / nc, j = e - i * nc;
        const double *Ci = T + tri(ns + i), *Cj = T + tri(ns + j);
        double s = 0.0;
        for (int k = lane; k < ns; k += 32) s = fma(Ci[k], Cj[k], s);
        s = warp_sum(s);
        if (lane == 0) S0[i * ncm + j] = Kcc[i * ncm + j] - s;
    }
    double part = 0.0;
    for (int i = tid; i < ns; i += NT) part = fma(u_s[i], ua_s[i], part);
    const double BA_S = block_sum2<NT>(part, red);
    __syncthreads();
    // small candidate-block solves (nc <= 16): thread 0
    if (tid == 0) {
        for (int i = 0; i < nc; ++i)
            for (int j = 0; j < nc; ++j) {
                M[lay.off_s0 + i * NC_MAX + j] = S0[i * ncm + j];
                M[lay.off_lcc0 + i * NC_MAX + j] = (j <= i) ? T[tri(ns + i) + ns + j] : 0.0;
            }
        for (int i = 0; i < nc; ++i) {   // ug0 = L_cc^-1 wb ; ua0 = L_cc^-1 wa
            double s1 = M[lay.off_wb + i], s2 = M[lay.off_wa + i];
            for (int k = 0; k < i; ++k) {
                const double l = T[tri(ns + i) + ns + k];
                s1 -= l * M[lay.off_ug0 + k];
                s2 -= l * M[lay.off_ua0 + k];
            }
            const double d = T[tri(ns + i) + ns + i];
            M[lay.off_ug0 + i] = s1 / d;
            M[lay.off_ua0 + i] = s2 / d;
            M[lay.off_rd0 + i] = 1.0 / d;
        }
        // alpha_c = L_cc^-T ua0  (back substitution)
        for (int i = nc - 1; i >= 0; --i) {
            double s = M[lay.off_ua0 + i];
            for (int k = i + 1; k < nc; ++k) s -= T[tri(ns + k) + ns + i] * alpha[ns + k];
            alpha[ns + i] = s / T[tri(ns + i) + ns + i];
        }
    }
    __syncthreads();
    PH(16);
    // ---- P11: alpha = K_l^-1 l_sc:  alpha_s = L_ss^-T (ua_s - C^T alpha_c)
    for (int i = tid; i < ns; i += NT) {
        double s = ua_s[i];
        for (int j = 0; j < nc; ++j) s -= T[tri(ns + j) + i] * alpha[ns + j];
        tmp[i] = s;
    }
    __syncthreads();
    lower_matvec_t_p<NT>(T, ns, tmp, alpha, nullptr, nullptr);
    PH(17);
    write_tri_frags<NT>(T, ns, c_l, M + lay.off_af_l_tri, lay.nb_cap);
    __syncthreads();
    // ---- s_l != 0: Z_mean / Z_var / log_lh use alpha_l = (K_l + s_l^2 I)^-1 l_sc (gp.inv_Kxx_y), while
    //      the bordered matrix above does not carry s_l^2 (SURVEY appendix A.2 asymmetry)
    if (s_l != 0.0) {
        for (int e = tid; e < tri(n); e += NT) {
            int i, j;
            tri_decode(e, i, j);
            double v = c_l * kernel_exp(x_sc[i] - x_sc[j], nh_l, kind, hp_l);
            if (i == j) v += s_l * s_l;
            T[e] = v;
        }
        __syncthreads();
        if (chol_packed<NT>(T, n, blk, &s_info, rdiag)) { if (tid == 0) M[H_STATUS] = SETUP_KL_NOTPD; return; }
        if (warp == 0) {   // forward then backward substitution, one warp
            for (int i = 0; i < n; ++i) {
                double s = 0.0;
                for (int k = lane; k < i; k += 32) s += T[tri(i) + k] * tmp2[k];
                s = warp_sum(s);
                if (lane == 0) tmp2[i] = (l_sc[i] - s) / T[tri(i) + i];
                __syncwarp();
            }
            for (int i = n - 1; i >= 0; --i) {
                double s = 0.0;
                for (int k = i + 1 + lane; k < n; k += 32) s += T[tri(k) + i] * alpha[k];
                s = warp_sum(s);
                if (lane == 0) alpha[i] = (tmp2[i] - s) / T[tri(i) + i];
                __syncwarp();
            }
        }
        __syncthreads();
        double p = 0.0;
        for (int i = tid; i < n; i += NT) p += log(T[tri(i) + i]);
        sumlog_l = block_sum2<NT>(p, red);
    }
    // alpha_l kept for the prediction kernel (bq_predict.cu): entry k belongs to x_sc[k], i.e. to M[off_xs + k] (k < ns) or
    // M[off_xc + k - ns]; zeros after n
    if (a.alpha) {
        double *ao = a.alpha + (size_t)inst * a.alpha_stride;
        for (int i = tid; i < a.alpha_stride; i += NT) ao[i] = i < n ? alpha[i] : 0.0;
    }
    PH(18);
    // ---- P12: Z_mean = int_K . alpha_l  (bq_c.pyx:207-209)
    double pz = 0.0;
    for (int i = tid; i < n; i += NT) pz = fma(b_sc[i], alpha[i], pz);
    double Zm = block_sum2<NT>(pz, red);
    // ---- P13: Z_var = alpha' M alpha - beta' K_tl^-1 beta  (bq_c.pyx:342-351)
    {
        double quad;                                            // first term; `beta` receives the vector of the second
        if (n_xo) {
            // trapezoid versions (bq.py:256-266, :315-327): m_j = gp_l.mean(xo_j), g_j = wp_j m_j,
            //   Z_mean = sum_j g_j                                                     bq_c.pyx:255-259
            //   Z_var  = g' K_tl(xo, xo) g - (K_tl(x_s, xo) g)' K_tl^-1 (K_tl(x_s, xo) g)    bq_c.pyx:404-420 with
            //            C_tl = gp_log_l.cov(xo) written out, so that the n_xo x n_xo matrix is never stored
            for (int j = tid; j < n_xo; j += NT) {
                const double xj = xo[j];
                double m = 0.0;
                for (int i = 0; i < n; ++i) m = fma(kernel_exp(xj - x_sc[i], nh_l, kind, hp_l), alpha[i], m);
                gz[j] = wp[j] * (c_l * m);
            }
            __syncthreads();
            double zp = 0.0;
            for (int j = tid; j < n_xo; j += NT) zp += gz[j];
            Zm = block_sum2<NT>(zp, red);
            double acc = 0.0;
            for (int i = warp; i < n_xo; i += NW) {
                const double xi = xo[i];
                double col = 0.0;
                for (int j = lane; j <= i; j += 32) {
                    const double kij = kernel_exp(xi - xo[j], nh_tl, kind, hp_tl);
                    col = fma(gz[j], j < i ? 2.0 * kij : kij, col);
                }
                col = warp_sum(col);
                if (lane == 0) acc = fma(col, gz[i], acc);
            }
            quad = c_tl * block_sum2<NT>(acc, red);
            for (int i = warp; i < ns; i += NW) {
                const double xi = x_sc[i];
                double r = 0.0;
                for (int j = lane; j < n_xo; j += 32) r = fma(kernel_exp(xi - xo[j], nh_tl, kind, hp_tl), gz[j], r);
                r = warp_sum(r);
                if (lane == 0) beta[i] = c_tl * r;
            }
            __syncthreads();
            PH(19);
        } else {
        //   M_ij = h_l^4 h_tl^2 exp(N1_i + N1_j + N2_ij)          gauss_c.pyx:488-529 (d = 1); symmetric, evaluated for i <= j
        const double A_ = sig2 * ((sig2 / Lb) / Lb);            // cov (W1 + cov)^-1 cov     :496-500
        const double C2 = w_tl * w_tl + 2 * sig2 - 2 * A_;     // :515
        const double L2 = sqrt(C2), logdet2 = 2 * log(L2), rL2 = 1.0 / L2;
        const double hh = (h_l * h_l * h_l * h_l) * (h_tl * h_tl);
        // B_i = cov (W1 + cov)^-1 x_i  -> tmp ; N1_i -> tmp2
        for (int i = tid; i < n; i += NT) {
            tmp[i] = sig2 * ((x_sc[i] / Lb) / Lb);
            tmp2[i] = mvn_logpdf1b(x_sc[i], mu, Lb, logdet_b);
        }
        __syncthreads();
        double acc = 0.0;
        for (int j = warp; j < n; j += NW) {
            double col = 0.0;
            const double bj = tmp[j], nj = tmp2[j];
            for (int i = lane; i <= j; i += 32) {
                const double mij = hh * exp(tmp2[i] + nj + mvn_logpdf1r(tmp[i], bj, rL2, logdet2));
                col += alpha[i] * (i < j ? 2.0 * mij : mij);
            }
            col = warp_sum(col);
            if (lane == 0) acc += col * alpha[j];
        }
        quad = block_sum2<NT>(acc, red);
        PH(19);
        //   int_K1_K2[i, j] = h_tl^2 h_l^2 N([x_s_i, x_sc_j] | [mu, mu], [[w_tl^2 + cov, cov], [cov, w_l^2 + cov]])
        //   gauss_c.pyx:305-337 with the 2 x 2 Cholesky done in closed form
        const double c00 = w_tl * w_tl + sig2, c11 = w_l * w_l + sig2;
        const double l00 = sqrt(c00), l10 = sig2 / l00, l11 = sqrt(c11 - l10 * l10);
        const double r00 = 1.0 / l00, r11 = 1.0 / l11;
        const double logdet12 = 2 * (log(l00) + log(l11));
        const double h12 = (h_tl * h_tl) * (h_l * h_l);
        for (int i = warp; i < ns; i += NW) {
            double s = 0.0;
            const double d0 = x_sc[i] - mu;
            const double y0 = d0 * r00;
            for (int j = lane; j < n; j += 32) {
                const double d1 = x_sc[j] - mu;
                // dpotrs: forward  y0 = d0/l00, y1 = (d1 - l10 y0)/l11 ; backward z1 = y1/l11, z0 = (y0 - l10 z1)/l00
                const double y1 = (d1 - l10 * y0) * r11;
                const double z1 = y1 * r11, z0 = (y0 - l10 * z1) * r00;
                const double lp = -0.5 * ((S2_LOG_2PI * 2 + logdet12) + (d0 * z0 + d1 * z1));
                s += (h12 * exp(lp)) * alpha[j];
            }
            s = warp_sum(s);
            if (lane == 0) beta[i] = s;
        }
        __syncthreads();
        }
        PH(20);
        // |L_tl^-1 beta|^2 = beta' K_tl^-1 beta, L_tl^-1 from its fragment-ordered copy (scaled by c_tl)
        double q = 0.0;
        {
            // a warp per row block: every fragment is one coalesced 256-byte read (lane l <-> row l >> 2, column l & 3),
            // the four lanes of a row are combined by two shuffles
            const double *F = M + lay.off_af_tl_tri;
            const int lc = lane & 3;
            for (int rb = warp; rb < (ns + 7) >> 3; rb += NW) {
                const double *Fb = F + ((size_t)(rb * (rb + 1)) << 5) + lane;
                const int nk = 2 * rb + 2;
                double s0 = 0.0, s1 = 0.0;
                for (int ks = 0; ks < nk; ks += 2) {
                    const int k0 = 4 * ks + lc, k1 = k0 + 4;
                    s0 = fma(Fb[ks << 5], k0 < ns ? beta[k0] : 0.0, s0);
                    s1 = fma(Fb[(ks + 1) << 5], k1 < ns ? beta[k1] : 0.0, s1);
                }
                double sr = s0 + s1;
                sr += __shfl_xor_sync(0xffffffffu, sr, 1);
                sr += __shfl_xor_sync(0xffffffffu, sr, 2);
                if (lc == 0) q = fma(sr, sr, q);
            }
        }
        const double beta2 = block_sum2<NT>(q, red) / (c_tl * c_tl);
        // ---- P14: log marginal likelihood of both GPs (bq.py:546; gp.log_lh)
        double y1 = 0.0, y2 = 0.0;
        for (int i = tid; i < ns; i += NT) y1 = fma(tl_s[i], a_tl[i], y1);
        for (int i = tid; i < n; i += NT) y2 = fma(l_sc[i], alpha[i], y2);
        const double yKy_tl = block_sum2<NT>(y1, red), yKy_l = block_sum2<NT>(y2, red);
        if (tid == 0) {
            M[H_ZM] = Zm;
            M[H_ZV] = quad - beta2;
            M[H_LOGLH] = (-0.5 * yKy_tl - sumlog_tl - 0.5 * ns * S2_LOG_2PI) + (-0.5 * yKy_l - sumlog_l - 0.5 * n * S2_LOG_2PI);
        }
    }
    PH(21);
    // ---- P15/P16: header and vectors
    double t2 = 0.0;
    for (int i = tid; i < ns; i += NT) { const double t = isclose_tol(x_sc[i]); t2 = fmax(t2, t * t); }
    t2 = block_max2<NT>(t2, red);
    if (tid == 0) {
        M[H_NS] = ns; M[H_NC] = nc; M[H_NSP] = nsp; M[H_STATUS] = SETUP_OK; M[H_NDB] = ndb;
        M[H_CL] = c_l; M[H_NHL] = -0.5 / (w_l * w_l); M[H_WL] = w_l;
        M[H_CTL] = c_tl; M[H_NHTL] = -0.5 / (w_tl * w_tl);
        // bq_c.pyx:136: jitter = max(EPS, np.max(M)) * 1e-4, np.max re-evaluated after the first pass
        const double j1 = fmax(EPS, c_l) * 1e-4;
        M[H_J1] = j1;
        M[H_KAA_E] = c_l + fmax(EPS, c_l) * 1e-4;
        M[H_KAA_N] = c_l + fmax(EPS, c_l + j1) * 1e-4;
        M[H_KTT] = c_tl;
        // isclose pre-filter of the scoring kernel: an upper bound of every tolerance squared
        M[H_TOL2MAX] = t2 * 1.000001;
        M[H_MU] = mu; M[H_THRESH] = thresh; M[H_BA_S] = BA_S;
        M[H_KIND] = kind; M[H_HP_TL] = hp_tl; M[H_HP_L] = hp_l;
        // int_K at a new point: h^2 exp(-1/2 (log 2pi + logdet)) * exp(-1/2 diff^2 / var)  (gauss_c.pyx:110, :162)
        M[H_CB] = (h_l * h_l) * exp(-0.5 * (S2_LOG_2PI + logdet_b)); M[H_NHB] = -0.5 / var_b;
    }
    for (int i = tid; i < lay.nsp_cap; i += NT) {
        const bool in = i < ns;
        M[lay.off_xs + i] = in ? x_sc[i] : 1e150;
        M[lay.off_tol + i] = in ? isclose_tol(x_sc[i]) : -1.0;
        M[lay.off_atl + i] = in ? c_tl * a_tl[i] : 0.0;
    }
    for (int i = tid; i < nc; i += NT) M[lay.off_xc + i] = x_sc[ns + i];
    PH(22);
#ifdef BQB_SETUP_PROF
    if (tid == 0 && blockIdx.x == 0) {
        printf("setup2<%d> ns=%d nc=%d phases (cycles):", NT, ns, nc);
        for (int i = 1; i <= 22; ++i) printf(" %d:%lld", i, s_prof[i] - s_prof[i - 1]);
        printf(" total %lld\n   chol: first diag %lld panel %lld column %lld diag|rest %lld ; inverse: stage %lld solve %lld\n", s_prof[22] - s_prof[0],
               g_s2_sub[0], g_s2_sub[1], g_s2_sub[2], g_s2_sub[5], g_s2_sub[3], g_s2_sub[4]);
    }
#endif
}

template <bool TSMEM, int NT, int KIND>
static cudaError_t launch_kind(const SetupArgs &a, int n_inst, size_t bytes, cudaStream_t stream) {
    cudaError_t e = cudaFuncSetAttribute(bq_setup2_kernel<TSMEM, NT, KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return e;
    bq_setup2_kernel<TSMEM, NT, KIND><<<n_inst, NT, bytes, stream>>>(a);
    return cudaGetLastError();
}
template <bool TSMEM, int NT>
static cudaError_t launch_one(const SetupArgs &a, int n_inst, size_t bytes, cudaStream_t stream) {
    return a.kind ? launch_kind<TSMEM, NT, 1>(a, n_inst, bytes, stream) : launch_kind<TSMEM, NT, 0>(a, n_inst, bytes, stream);
}

// opt-in maximum of dynamic shared memory per CTA minus the kernel's static shared memory
constexpr size_t S2_CTA_SMEM_MAX = 227 * 1024 - 256;

// Largest instance order n for which two 256-thread CTAs of the setup kernel fit one SM (0: none), given the launch's nc_max.
int setup2_two_cta_limit(int nc_max) {
    static int cache[NC_MAX + 2];
    static bool have[NC_MAX + 2];
    if (nc_max < 0 || nc_max > NC_MAX) return 0;
    if (have[nc_max]) return cache[nc_max];
    int lo = 0, hi = 218;                              // invariant: lo fits (or is 0), hi + 1 does not
    while (lo < hi) {
        const int mid = (lo + hi + 1) / 2;
        const size_t bytes = sizeof(double) * (size_t)s2_carve(mid, nc_max, true).total;
        int per_sm = 0;
        bool ok = bytes <= S2_CTA_SMEM_MAX &&
                  cudaFuncSetAttribute(bq_setup2_kernel<true, 256, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) == cudaSuccess &&
                  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bq_setup2_kernel<true, 256, 0>, 256, bytes) == cudaSuccess && per_sm >= 2;
        if (ok) lo = mid; else hi = mid - 1;
    }
    cudaGetLastError();
    have[nc_max] = true;
    return cache[nc_max] = lo;
}

// Global scratch (doubles per instance, SetupArgs::work_stride) that launch_setup2 can need for instances of capacity
// class cap: 0 when the largest instance (cap observations, NC_MAX candidates) keeps its triangle in shared memory, else
// the stride of a packed triangle of that order.
size_t setup2_scratch_stride(int cap) {
    const int n = cap + NC_MAX;
    if (sizeof(double) * (size_t)s2_carve(n, NC_MAX, true).total <= S2_CTA_SMEM_MAX) return 0;
    return ((size_t)n * (n + 1) / 2 + 64) & ~(size_t)1;
}

// a.n_max / a.nc_max must be >= ns + nc / nc of every instance of the launch (instances above report SETUP_BAD_INPUT)
cudaError_t launch_setup2(const SetupArgs &a, int n_inst, cudaStream_t stream) {
    const size_t bytes_sm = sizeof(double) * (size_t)s2_carve(a.n_max, a.nc_max, true).total;
    if (bytes_sm <= S2_CTA_SMEM_MAX) {
        // two CTAs of 256 threads per SM when two instances fit (their serial phases overlap), else one of 512
        int per_sm = 0;
        cudaError_t e = cudaFuncSetAttribute(bq_setup2_kernel<true, 256, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes_sm);
        if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bq_setup2_kernel<true, 256, 0>, 256, bytes_sm);
        if (e != cudaSuccess) return e;
        // (a launch that does not fill the SMs once is a latency problem, not a throughput one: 512 threads per instance)
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (per_sm >= 2 && n_inst > sms) return launch_one<true, 256>(a, n_inst, bytes_sm, stream);
        return launch_one<true, 512>(a, n_inst, bytes_sm, stream);
    }
    const size_t bytes = sizeof(double) * (size_t)s2_carve(a.n_max, a.nc_max, false).total;
    return launch_one<false, 512>(a, n_inst, bytes, stream);
}

// ============================================================================================================================
// Value and gradient of the joint log marginal likelihood ll = ll_tl + ll_l (BQ._make_llh_params, bq.py:533-552) with
// respect to the hyper-parameters, one CTA per (instance, hyper-parameter row).  KIND 0: gp.GaussianKernel, six
// derivatives; KIND 1: gp.PeriodicKernel, eight (the periods p_tl and p_l last).
//
//   ll_tl: gp_log_l on (x_s, log l_s), K_t = c_t E_t + s_t^2 I, c = h^2 / (sqrt(2 pi) w), E_ij = exp(-d_ij^2 / 2 w^2)
//   ll_l:  gp_l on (x_sc, [l_s; l_c]), K_l = c_l E_l + s_l^2 I, l_c[j] = exp(m_j), m_j = k_j' a, a = K_t^-1 log l_s
//   d ll / d theta_l = 1/2 alpha' Kd alpha - 1/2 tr(K_l^-1 Kd),   alpha = K_l^-1 l_sc
//   d ll / d theta_t = 1/2 a' Kd a - 1/2 tr(K_t^-1 Kd) - sum_j gamma_j dm_j,   gamma_j = alpha[ns + j] l_c[j]
//       dm_j = kd_j' a - k_j' K_t^-1 Kd a
//   Kd_h = 2 G / h, Kd_w = G . D^2 / w^3 - G / w, Kd_s = 2 s I  (G = c E; kd_j the same for the cross-kernel, kd_s = 0)
//   tr(K^-1 Kd_h) = 2 (n - s^2 tr K^-1) / h,  tr(K^-1 Kd_s) = 2 s tr K^-1,  tr K^-1 = |L^-1|_F^2
//   tr(K^-1 Kd_w) = sum_ij (K^-1)_ij G_ij d_ij^2 / w^3 - (n - s^2 tr K^-1) / w
//
// Storage: one packed triangle serves both GPs, as in the setup kernel (the same carve-up, s2_carve, plus three vectors
// and the 3 x nc derivatives dm_j).  tl phase: L_t -> L_t^-1 in place, a, l_c, the guard, the tl traces, and dm_j for
// every candidate and tl parameter from the three vectors K_t^-1 G a, K_t^-1 (G . D^2) a and K_t^-1 a (so no ns x nc
// matrix is kept).  l phase: L_l -> L_l^-1 in place, alpha, the l traces; then the -sum gamma_j dm_j terms.  The only
// trace that needs entries of K^-1 (the w-trace) evaluates (K^-1)_ij = sum_{k >= i} X_ki X_kj (X = L^-1) for i > j, one
// thread per entry, and never stores them.
//
// Periodic kernel (KIND 1): K = c exp(nh D^2) with c = h^2 (independent of w), nh = -1 / (2 w^2), D = 2 sin(d / 2p), and
// F_ij = d_ij sin(d_ij / p) / (w^2 p^2):
//   Kd_h = 2 G / h, Kd_w = G . D^2 / w^3 (no -G / w term), Kd_p = G . F (one per GP), Kd_s = 2 s I
//   tr(K^-1 Kd_p) = sum_ij (K^-1)_ij G_ij F_ij, accumulated in the pass of the w-trace from the same (K^-1)_ij
//   dm_j / dp_tl = (k_j . F(x_c[j] - x_s))' a - k_j' K_t^-1 (G . F) a
// which needs a fourth live vector K_t^-1 (G . F) a and a fourth row of dm_j.
//
// Observations are sorted as in the setup kernel, and the tl factor, a and l_c are computed by the same code, so l_c and
// the guard are the setup's bit for bit.  Every reduction has a fixed order and the CTA shape is fixed (256 threads), so
// a row's results do not depend on the other rows of the launch.  Status codes and the order of the checks are the
// setup's: a K_l without the noise s_l^2 that is not positive definite is SETUP_KL_NOTPD even when s_l != 0.
constexpr int LLG_NT = 256;
constexpr int LLG_NVEC = 3;     // K_t^-1 G a, K_t^-1 (G . D^2) a, K_t^-1 a: live across the candidate pass (stage)

// kind 1 adds the vector K_t^-1 (G . F) a and the row dm_j / dp_tl
__host__ __device__ inline int llg_smem_doubles(int nmax, int ncm, bool tsmem, int kind) {
    const S2Carve c = s2_carve(nmax, ncm, tsmem);
    return c.total + (LLG_NVEC + kind) * c.nv + (3 + kind) * NC_MAX;
}

// D^2 = (2 sin(d hp))^2 and F = d sin(d / p) / (w^2 p^2) of the periodic kernel (hp = 1 / (2 p), nh = -1 / (2 w^2))
__device__ __forceinline__ void llg_periodic_terms(double d, double nh, double hp, double &D2, double &F) {
    double sn, cs;
    sincos(d * hp, &sn, &cs);
    D2 = (2.0 * sn) * (2.0 * sn);
    F = d * (2.0 * sn * cs) * (-2.0 * nh) * (4.0 * hp * hp);
}

// sum over i > j of (K^-1)_ij G_ij D_ij^2 with K^-1 = X' X, X = L^-1 packed in T (partial sum of the calling thread);
// KIND 1 also sums (K^-1)_ij G_ij F_ij into *pp
template <int KIND>
__device__ __forceinline__ double llg_wtrace_part(const double *T, int n, const double *x, double c, double nh, double hp, double *pp) {
    double p = 0.0, q = 0.0;
    for (int e = threadIdx.x; e < tri(n); e += LLG_NT) {
        int i, j;
        tri_decode(e, i, j);
        if (j == i) continue;
        double kij = 0.0;
        for (int k = i, r = tri(i); k < n; r += ++k) kij = fma(T[r + i], T[r + j], kij);
        const double d = x[i] - x[j];
        if (KIND) {
            double D2, F;
            llg_periodic_terms(d, nh, hp, D2, F);
            const double g = c * kernel_exp(d, nh, 1, hp);
            p = fma(kij, g * D2, p);
            q = fma(kij, g * F, q);
        } else {
            const double d2 = d * d;
            p = fma(kij, c * kernel_exp(d, nh, 0, 0.0) * d2, p);
        }
    }
    if (KIND) *pp = q;
    return p;
}

// g1 = G v, g2 = (G . D^2) v (and for KIND 1 g3 = (G . F) v) over the first n points of x, a thread per row (G = c E,
// without the noise)
template <int KIND>
__device__ __forceinline__ void llg_gram_matvec(const double *x, int n, double c, double nh, double hp, const double *v, double *g1,
                                                double *g2, double *g3) {
    for (int i = threadIdx.x; i < n; i += LLG_NT) {
        double s1 = 0.0, s2 = 0.0, s3 = 0.0;
        for (int j = 0; j < n; ++j) {
            const double d = x[i] - x[j];
            const double g = c * kernel_exp(d, nh, KIND, hp);
            s1 = fma(g, v[j], s1);
            if (KIND) {
                double D2, F;
                llg_periodic_terms(d, nh, hp, D2, F);
                s2 = fma(g * D2, v[j], s2);
                s3 = fma(g * F, v[j], s3);
            } else {
                s2 = fma(g * (d * d), v[j], s2);
            }
        }
        g1[i] = s1;
        g2[i] = s2;
        if (KIND) g3[i] = s3;
    }
    __syncthreads();
}

template <bool TSMEM, int KIND>
__global__ void __launch_bounds__(LLG_NT) bq_llgrad_kernel(LLGradArgs a) {
    constexpr int NT = LLG_NT, NW = NT / 32;
    constexpr int NOUT = KIND ? LLG_OUT_PERIODIC : LLG_OUT;
    __shared__ double red[NW];
    __shared__ int s_fail, s_info;
    extern __shared__ double s_dyn[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int e = a.e0 + blockIdx.x;
    const int inst = a.inst ? a.inst[e] : e;
    double *out = a.out + (size_t)e * NOUT;
    const int ns = a.ns[inst], nc = a.nc[inst], n = ns + nc;

    // carve-up: the setup kernel's, then [p1 p2 p3 (p4)] [dm (3 | 4) x NC_MAX]
    const S2Carve cv = s2_carve(a.n_max, a.nc_max, TSMEM);
    const int lds = cv.lds, nv = cv.nv;
    double *T = TSMEM ? s_dyn : a.work + (size_t)blockIdx.x * a.work_stride;
    double *vec = s_dyn + cv.np;
    double *tl_s = vec, *a_tl = vec + nv, *x_sc = vec + 2 * nv, *l_sc = vec + 3 * nv, *rdiag = vec + 4 * nv;
    double *un = vec + S2_NVEC_FIXED * nv;
    double *stage = un;
    double *u0 = un, *u1 = un + nv, *u2 = un + 2 * nv, *u3 = un + 3 * nv;
    double *u4 = un + 4 * nv, *u5 = un + 5 * nv;       // KIND 1 only
    double *blk = un + cv.un;
    double *p1 = s_dyn + cv.total, *p2 = p1 + nv, *p3 = p2 + nv;
    double *p4 = p3 + nv;                               // KIND 1 only: K_t^-1 (G . F) a
    double *dm = p3 + (KIND ? 2 : 1) * nv;

    auto fail = [&](int status) {
        if (tid == 0) {
            out[0] = -INFINITY;
            for (int k = 1; k < NOUT - 1; ++k) out[k] = NAN;
            out[NOUT - 1] = status;
        }
    };
    const double *hp = a.hyp + (size_t)e * 6;
    const double h_tl = hp[0], w_tl = hp[1], s_tl = hp[2], h_l = hp[3], w_l = hp[4], s_l = hp[5];
    const double p_tl = KIND ? a.period[(size_t)e * 2] : 0.0, p_l = KIND ? a.period[(size_t)e * 2 + 1] : 0.0;
    if (!(ns >= 1 && ns <= a.in_stride && nc >= 0 && nc <= NC_MAX && nc <= a.nc_max && n <= a.n_max)) { fail(SETUP_BAD_INPUT); return; }
    if (tid == 0) s_fail = SETUP_OK;
    __syncthreads();
    {
        const double *x_s = a.x_s + (size_t)inst * a.in_stride;
        const double *l_s = a.l_s + (size_t)inst * a.in_stride;
        const double *x_c = a.x_c + (size_t)inst * NC_MAX;
        int bad = 0;
        for (int i = tid; i < ns; i += NT) {
            const double x = x_s[i], l = l_s[i];
            bad |= !(isfinite(x) && isfinite(l) && l > 0.0);
            u0[i] = x;
            u1[i] = l;
        }
        for (int i = tid; i < nc; i += NT) {
            const double x = x_c[i];
            bad |= !isfinite(x);
            x_sc[ns + i] = x;
        }
        if (tid == 0) {
            for (int k = 0; k < 6; ++k) bad |= !isfinite(hp[k]);
            bad |= !(h_tl > 0 && w_tl > 0 && s_tl >= 0 && h_l > 0 && w_l > 0 && s_l >= 0);
            if (KIND) bad |= !(isfinite(p_tl) && isfinite(p_l) && p_tl > 0 && p_l > 0);
        }
        if (bad) s_fail = SETUP_BAD_INPUT;
    }
    __syncthreads();
    if (s_fail) { fail(s_fail); return; }
    // observations in ascending order of x, stable (the setup kernel's order)
    for (int i = tid; i < ns; i += NT) {
        const double xi = u0[i];
        int rank = 0;
        for (int j = 0; j < ns; ++j) {
            const double xj = u0[j];
            rank += (xj < xi) || (xj == xi && j < i);
        }
        x_sc[rank] = xi;
        l_sc[rank] = u1[i];
    }
    __syncthreads();

    // the setup kernel's expressions (bit for bit the same l_c and guard)
    const double hp_tl = KIND ? 0.5 / p_tl : 0.0, hp_l = KIND ? 0.5 / p_l : 0.0;
    const double c_tl = KIND ? h_tl * h_tl : (h_tl * h_tl) / (S2_SQRT_2PI * w_tl), nh_tl = -0.5 / (w_tl * w_tl);
    const double c_l = KIND ? h_l * h_l : (h_l * h_l) / (S2_SQRT_2PI * w_l), nh_l = -0.5 / (w_l * w_l);

    // ---- tl phase: K_t -> L_t -> L_t^-1, a
    for (int i = tid; i < ns; i += NT) tl_s[i] = log(l_sc[i]);
    for (int q = tid; q < tri(ns); q += NT) {
        int i, j;
        tri_decode(q, i, j);
        double v = c_tl * kernel_exp(x_sc[i] - x_sc[j], nh_tl, KIND, hp_tl);
        if (i == j) v += s_tl * s_tl;
        T[q] = v;
    }
    __syncthreads();
    if (chol_packed<NT>(T, ns, blk, &s_info, rdiag)) { fail(SETUP_KTL_NOTPD); return; }
    double sumlog_tl;
    {
        double p = 0.0;
        for (int i = tid; i < ns; i += NT) p += log(T[tri(i) + i]);
        sumlog_tl = block_sum2<NT>(p, red);
    }
    tri_inverse_packed<NT>(T, ns, stage, lds, rdiag);
    lower_matvec_p<NT>(T, ns, tl_s, u0, nullptr, nullptr);
    lower_matvec_t_p<NT>(T, ns, u0, a_tl, nullptr, nullptr);
    // u0 = G a, u1 = (G . D^2) a (u4 = (G . F) a); p1 = K_t^-1 u0, p2 = K_t^-1 u1, p3 = K_t^-1 a (p4 = K_t^-1 u4)
    llg_gram_matvec<KIND>(x_sc, ns, c_tl, nh_tl, hp_tl, a_tl, u0, u1, u4);
    lower_matvec_p<NT>(T, ns, u0, u2, u1, u3);
    lower_matvec_t_p<NT>(T, ns, u2, p1, u3, p2);
    lower_matvec_p<NT>(T, ns, a_tl, u2, KIND ? u4 : nullptr, KIND ? u5 : nullptr);
    lower_matvec_t_p<NT>(T, ns, u2, p3, KIND ? u5 : nullptr, KIND ? p4 : nullptr);
    double g_tl[4], yKy_tl;
    {
        double pg1 = 0.0, pg2 = 0.0, paa = 0.0, py = 0.0, ptr = 0.0, pg3 = 0.0, pp = 0.0;
        for (int i = tid; i < ns; i += NT) {
            pg1 = fma(a_tl[i], u0[i], pg1);
            pg2 = fma(a_tl[i], u1[i], pg2);
            paa = fma(a_tl[i], a_tl[i], paa);
            if (KIND) pg3 = fma(a_tl[i], u4[i], pg3);
        }
        for (int i = tid; i < ns; i += NT) py = fma(tl_s[i], a_tl[i], py);
        for (int q = tid; q < tri(ns); q += NT) ptr = fma(T[q], T[q], ptr);
        const double aga = block_sum2<NT>(pg1, red), agda = block_sum2<NT>(pg2, red), aa = block_sum2<NT>(paa, red);
        yKy_tl = block_sum2<NT>(py, red);
        const double trK = block_sum2<NT>(ptr, red);
        const double wtr = 2.0 * block_sum2<NT>(llg_wtrace_part<KIND>(T, ns, x_sc, c_tl, nh_tl, hp_tl, &pp), red);
        const double rest = ns - s_tl * s_tl * trK;
        g_tl[0] = (aga - rest) / h_tl;
        if (KIND) {
            g_tl[1] = 0.5 * (agda - wtr) / (w_tl * w_tl * w_tl);
            const double agfa = block_sum2<NT>(pg3, red), ptrace = 2.0 * block_sum2<NT>(pp, red);
            g_tl[3] = 0.5 * (agfa - ptrace);
        } else {
            g_tl[1] = 0.5 * ((agda - wtr) / (w_tl * w_tl * w_tl) - (aga - rest) / w_tl);
        }
        g_tl[2] = s_tl * (aa - trK);
    }
    // l_c = exp(k_j' a), the guard and dm_j, four candidates per pass (the setup kernel's P6, plus the three dm_j):
    // stage rows 0..3 = k_j, rows 4..7 = (L_t^-1 k_j)^2 element-wise (the guard only)
    for (int j0 = 0; j0 < nc; j0 += 4) {
        const int nbt = (nc - j0 < 4) ? nc - j0 : 4;
        for (int q = tid; q < nbt * ns; q += NT) {
            const int j = q / ns, k = q - j * ns;
            stage[j * lds + k] = c_tl * kernel_exp(x_sc[ns + j0 + j] - x_sc[k], nh_tl, KIND, hp_tl);
        }
        __syncthreads();
        if (a.check_max) {
            for (int q = tid; q < nbt * ns; q += NT) {
                const int j = q / ns, r = q - j * ns;
                const double *row = T + tri(r), *kc = stage + j * lds;
                double s0 = 0.0, s1 = 0.0;
                int k = 0;
                for (; k + 1 <= r; k += 2) {
                    s0 = fma(row[k], kc[k], s0);
                    s1 = fma(row[k + 1], kc[k + 1], s1);
                }
                if (k <= r) s0 = fma(row[k], kc[k], s0);
                const double y = s0 + s1;
                stage[(4 + j) * lds + r] = y * y;
            }
            __syncthreads();
        }
        if (warp < nbt) {
            const int j = warp;
            const double xc = x_sc[ns + j0 + j];
            double m = 0.0, q = 0.0, r = 0.0, q1 = 0.0, q2 = 0.0, q3 = 0.0, rp = 0.0, q4 = 0.0;
            for (int k = lane; k < ns; k += 32) {
                const double kv = stage[j * lds + k], d = xc - x_sc[k];
                m = fma(kv, a_tl[k], m);
                if (a.check_max) q += stage[(4 + j) * lds + k];
                if (KIND) {
                    double D2, F;
                    llg_periodic_terms(d, nh_tl, hp_tl, D2, F);
                    r = fma(kv * D2, a_tl[k], r);
                    rp = fma(kv * F, a_tl[k], rp);
                    q4 = fma(kv, p4[k], q4);
                } else {
                    r = fma(kv * (d * d), a_tl[k], r);
                }
                q1 = fma(kv, p1[k], q1);
                q2 = fma(kv, p2[k], q2);
                q3 = fma(kv, p3[k], q3);
            }
            m = warp_sum(m);
            q = warp_sum(q);
            r = warp_sum(r);
            q1 = warp_sum(q1);
            q2 = warp_sum(q2);
            q3 = warp_sum(q3);
            if (KIND) {
                rp = warp_sum(rp);
                q4 = warp_sum(q4);
            }
            if (lane == 0) {
                if (a.check_max) {
                    double V = c_tl - q;
                    if (V < 0) V = 0;
                    if (m + 2 * sqrt(V) > MAX_EXPONENT) s_fail = SETUP_MEAN_TOO_LARGE;
                }
                l_sc[ns + j0 + j] = exp(m);
                dm[j0 + j] = 2.0 * (m - q1) / h_tl;
                if (KIND) {
                    dm[NC_MAX + j0 + j] = (r - q2) / (w_tl * w_tl * w_tl);
                    dm[3 * NC_MAX + j0 + j] = rp - q4;
                } else {
                    dm[NC_MAX + j0 + j] = (r - q2) / (w_tl * w_tl * w_tl) - (m - q1) / w_tl;
                }
                dm[2 * NC_MAX + j0 + j] = -2.0 * s_tl * q3;
            }
        }
        __syncthreads();
    }
    __syncthreads();
    if (s_fail) { fail(s_fail); return; }

    // ---- l phase: K_l (the noise-free matrix first, as the setup kernel factorises it) -> L_l -> L_l^-1, alpha
    for (int pass = 0; pass < (s_l != 0.0 ? 2 : 1); ++pass) {
        for (int q = tid; q < tri(n); q += NT) {
            int i, j;
            tri_decode(q, i, j);
            double v = c_l * kernel_exp(x_sc[i] - x_sc[j], nh_l, KIND, hp_l);
            if (pass && i == j) v += s_l * s_l;
            T[q] = v;
        }
        __syncthreads();
        if (chol_packed<NT>(T, n, blk, &s_info, rdiag)) { fail(SETUP_KL_NOTPD); return; }
    }
    double sumlog_l;
    {
        double p = 0.0;
        for (int i = tid; i < n; i += NT) p += log(T[tri(i) + i]);
        sumlog_l = block_sum2<NT>(p, red);
    }
    tri_inverse_packed<NT>(T, n, stage, lds, rdiag);
    double *alpha = u1;
    lower_matvec_p<NT>(T, n, l_sc, u0, nullptr, nullptr);
    lower_matvec_t_p<NT>(T, n, u0, alpha, nullptr, nullptr);
    llg_gram_matvec<KIND>(x_sc, n, c_l, nh_l, hp_l, alpha, u2, u3, u4);
    {
        double pg1 = 0.0, pg2 = 0.0, paa = 0.0, py = 0.0, ptr = 0.0, pg3 = 0.0, pp = 0.0;
        for (int i = tid; i < n; i += NT) {
            pg1 = fma(alpha[i], u2[i], pg1);
            pg2 = fma(alpha[i], u3[i], pg2);
            paa = fma(alpha[i], alpha[i], paa);
            if (KIND) pg3 = fma(alpha[i], u4[i], pg3);
        }
        for (int i = tid; i < n; i += NT) py = fma(l_sc[i], alpha[i], py);
        for (int q = tid; q < tri(n); q += NT) ptr = fma(T[q], T[q], ptr);
        const double aga = block_sum2<NT>(pg1, red), agda = block_sum2<NT>(pg2, red), aa = block_sum2<NT>(paa, red);
        const double yKy = block_sum2<NT>(py, red), trK = block_sum2<NT>(ptr, red);
        const double wtr = 2.0 * block_sum2<NT>(llg_wtrace_part<KIND>(T, n, x_sc, c_l, nh_l, hp_l, &pp), red);
        double agfa = 0.0, ptrace = 0.0;
        if (KIND) {
            agfa = block_sum2<NT>(pg3, red);
            ptrace = 2.0 * block_sum2<NT>(pp, red);
        }
        if (tid == 0) {
            const double rest = n - s_l * s_l * trK;
            double ch = 0.0, cw = 0.0, cs = 0.0, cp = 0.0;        // sum_j gamma_j dm_j, in candidate order
            for (int j = 0; j < nc; ++j) {
                const double gam = alpha[ns + j] * l_sc[ns + j];
                ch = fma(gam, dm[j], ch);
                cw = fma(gam, dm[NC_MAX + j], cw);
                cs = fma(gam, dm[2 * NC_MAX + j], cs);
                if (KIND) cp = fma(gam, dm[3 * NC_MAX + j], cp);
            }
            out[0] = (-0.5 * yKy_tl - sumlog_tl - 0.5 * ns * S2_LOG_2PI) + (-0.5 * yKy - sumlog_l - 0.5 * n * S2_LOG_2PI);
            out[1] = g_tl[0] - ch;
            out[2] = g_tl[1] - cw;
            out[3] = g_tl[2] - cs;
            out[4] = (aga - rest) / h_l;
            if (KIND) {
                out[5] = 0.5 * (agda - wtr) / (w_l * w_l * w_l);
                out[6] = s_l * (aa - trK);
                out[7] = g_tl[3] - cp;
                out[8] = 0.5 * (agfa - ptrace);
            } else {
                out[5] = 0.5 * ((agda - wtr) / (w_l * w_l * w_l) - (aga - rest) / w_l);
                out[6] = s_l * (aa - trK);
            }
            out[NOUT - 1] = SETUP_OK;
        }
    }
}

template <bool TSMEM, int KIND>
static cudaError_t launch_llgrad_one(const LLGradArgs &a, int n_rows, size_t bytes, cudaStream_t stream) {
    cudaError_t e = cudaFuncSetAttribute(bq_llgrad_kernel<TSMEM, KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return e;
    bq_llgrad_kernel<TSMEM, KIND><<<n_rows, LLG_NT, bytes, stream>>>(a);
    return cudaGetLastError();
}

template <int KIND>
static cudaError_t launch_llgrad_kind(LLGradArgs a, int n_rows, int work_inst, cudaStream_t stream, int *launches) {
    const size_t bytes_sm = sizeof(double) * (size_t)llg_smem_doubles(a.n_max, a.nc_max, true, KIND);
    *launches = 0;
    if (bytes_sm <= S2_CTA_SMEM_MAX) {
        *launches = 1;
        return launch_llgrad_one<true, KIND>(a, n_rows, bytes_sm, stream);
    }
    const int n_big = a.n_max;
    if (!a.work || a.work_stride < (size_t)tri(n_big) || work_inst < 1) return cudaErrorInvalidValue;
    const size_t bytes = sizeof(double) * (size_t)llg_smem_doubles(a.n_max, a.nc_max, false, KIND);
    const int end = a.e0 + n_rows;
    for (int e0 = a.e0; e0 < end; e0 += work_inst) {
        a.e0 = e0;
        cudaError_t e = launch_llgrad_one<false, KIND>(a, end - e0 < work_inst ? end - e0 : work_inst, bytes, stream);
        ++*launches;
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// Rows [a.e0, a.e0 + n_rows) of kernel kind 0 (Gaussian) or 1 (periodic, a.period set): one launch while the triangle fits
// shared memory, else launches of at most work_inst CTAs on the global scratch a.work (work_inst triangles of a.work_stride
// doubles).  *launches counts the kernel launches.
cudaError_t launch_llgrad(LLGradArgs a, int n_rows, int work_inst, cudaStream_t stream, int *launches, int kind) {
    return kind ? launch_llgrad_kind<1>(a, n_rows, work_inst, stream, launches)
                : launch_llgrad_kind<0>(a, n_rows, work_inst, stream, launches);
}

}  // namespace bqb
