// Generic scoring kernel: the same per-point border update as bq_score.cu for the cases its tensor-core kernels do not
// cover -- gp.PeriodicKernel (no band structure: sin^2 does not decay) and the reference's trapezoid approximation of
// int_K for non-Gaussian kernels (`use_approx`, bq.py:498-510 -> bq_c.approx_expected_squared_mean_and_mean
// bq_c.pyx:538-598: int_K[i] = trapz(K_l(x_i, xo) p(xo))).
//
// A CTA of eight warps works on a tile of 32 query points, lane = point, plain FP64: the cross-kernel vectors of the 32
// points are kept in shared memory ([k][lane], conflict free) and shared by the warps, which split the rows of c L^-1
// (fragment order, as the tensor-core kernels read them; warp-uniform 16-byte loads from global memory), the dense rows, the
// fill of the cross-kernel vectors and the trapezoid sum; warp 0 combines the partial sums in a fixed order and runs the
// per-point tail.  (The first version gave every point ONE thread and a warp its own [k][32] buffer: one warp per SM at 512
// observations, 59 % of the stall samples on the operand loads, FP64 pipe 1.5 % busy -- profiles/ncu_generic_r02.md.)  This is the reference's *slow* path (its own cost is n_xo = 1000 kernel evaluations per query
// point in a Python loop); the kernel is meant to be correct and complete, not at a roofline: ~n^2 FMA + n_xo
// kernel evaluations per point.  With the Gaussian kernel and n_xo = 0 it computes exactly what bq_score.cu computes
// (dense algorithm), which is how tests/test_gpu_generic.py validates it.
#include "bq_common.cuh"

namespace bqb {

constexpr int GEN_THREADS = 32;              // points per tile (= lanes)
constexpr int GEN_WARPS = 8;                 // warps of a CTA: they share the tile
constexpr int GEN_MAX_GRID = 2048;            // the fused epilogue leaves one (min, index) partial per CTA

// sum_{k <= r} F[r][k] e[k] for row r of a triangular fragment-ordered operand: a k-step is four consecutive doubles of the
// row (32-byte aligned: two 16-byte warp-uniform loads); entries with k > r are stored as zeros, so whole k-steps are used
// (the e buffer is zero for k >= ns)
__device__ __forceinline__ double tri_row_dot(const double *F, int r, const double *s_e, int lane) {
    const int rb = r >> 3;
    const double2 *row = reinterpret_cast<const double2 *>(F + ((rb * (rb + 1)) << 5) + ((r & 7) << 2));
    const double *e = s_e + lane;
    double s0 = 0.0, s1 = 0.0;
    for (int ks = 0; ks <= (r >> 2); ++ks) {
        const double2 f01 = row[ks << 4], f23 = row[(ks << 4) + 1];
        const double *ek = e + (ks << 2) * GEN_THREADS;
        s0 = fma(f01.x, ek[0], s0);
        s1 = fma(f01.y, ek[GEN_THREADS], s1);
        s0 = fma(f23.x, ek[2 * GEN_THREADS], s0);
        s1 = fma(f23.y, ek[3 * GEN_THREADS], s1);
    }
    return s0 + s1;
}

__global__ void __launch_bounds__(GEN_THREADS * GEN_WARPS) bq_score_generic_kernel(ScoreArgs a) {
    extern __shared__ double s_e[];                                  // [nsp][32] cross-kernel exponentials of the tile's points
    __shared__ double s_dr[NC_MAX + 2][GEN_THREADS];                 // dense rows / v_c
    __shared__ double s_part[4][GEN_WARPS][GEN_THREADS];             // per-warp partial sums: qs, qt, tm, int_K at the point
    __shared__ int s_close[GEN_WARPS][GEN_THREADS];
    const Layout lay = a.lay;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int inst = a.inst0 + blockIdx.y;
    const double *M = a.models + (size_t)inst * lay.total;
    const int ns = (int)M[H_NS], nc = (int)M[H_NC], nsp = (int)M[H_NSP];
    const int nks = nsp >> 2;
    const int kind = (int)M[H_KIND];
    const double hp_tl = M[H_HP_TL], hp_l = M[H_HP_L];
    const double c_l = M[H_CL], nhl = M[H_NHL], nhtl = M[H_NHTL];
    const double Zm = M[H_ZM];
    const double *xs = M + lay.off_xs, *tol = M + lay.off_tol, *atl = M + lay.off_atl, *xc = M + lay.off_xc;
    const double *Fl = M + lay.off_af_l_tri, *Fd = M + lay.off_af_l_dense, *Ft = M + lay.off_af_tl_tri;
    const double *xa = a.x_a + (size_t)(inst / a.xa_group) * a.xa_stride;
    double *o_esm = a.esm ? a.esm + (size_t)inst * a.out_stride : nullptr;
    double *o_em = a.em ? a.em + (size_t)inst * a.out_stride : nullptr;
    int *o_st = a.status ? a.status + (size_t)inst * a.out_stride : nullptr;
    const double *xo = a.n_xo ? a.xo + (size_t)inst * a.xo_stride : nullptr;
    const double *wp = a.n_xo ? a.wp + (size_t)inst * a.n_xo : nullptr;
    const bool epi = a.ev != nullptr;

    double best_v = INFINITY;
    long long best_i = 0x7fffffffffffffffLL;
    int cta_st = 0;
    if (warp == 0)
        for (int k = ns; k < nsp; ++k) s_e[k * GEN_THREADS + lane] = 0.0;  // padding of the last k-step
    for (long long t0 = (long long)blockIdx.x * GEN_THREADS; t0 < a.na; t0 += (long long)gridDim.x * GEN_THREADS) {
        const long long p = t0 + lane;
        const bool live = p < a.na;
        const double xv = live ? xa[p] : 0.0;
        const bool fin = live && isfinite(xv);
        const double x = fin ? xv : 0.0;
        // ---- K_l pass: e[k] = exp part of K_l(x, x_s[k]);  v_s = (c_l L_ss^-1) e,  dense rows (c_l [W; g_gamma; g_alpha]) e
        __syncthreads();                                                  // the previous tile's tail has left s_dr / s_part
        int close_w = 0;
        for (int k = warp; k < ns; k += GEN_WARPS) {
            const double d = x - xs[k];
            close_w |= fabs(d) <= tol[k];                                 // np.isclose(x_a, x_s, atol = 1e-4)  bq.py:456
            s_e[k * GEN_THREADS + lane] = kernel_exp(d, nhl, kind, hp_l);
        }
        s_close[warp][lane] = close_w;
        __syncthreads();
        double qs = 0.0;
        for (int r = warp; r < ns; r += GEN_WARPS) {
            const double v = tri_row_dot(Fl, r, s_e, lane);
            qs = fma(v, v, qs);
        }
        s_part[0][warp][lane] = qs;
        for (int r = warp; r < nc + 2; r += GEN_WARPS) {
            const double2 *row = reinterpret_cast<const double2 *>(Fd + (((r >> 3) * nks) << 5) + ((r & 7) << 2));
            double s0 = 0.0, s1 = 0.0;
            for (int ks = 0; ks < nks; ++ks) {                     // columns k >= ns are stored as zeros
                const double2 f01 = row[ks << 4], f23 = row[(ks << 4) + 1];
                const double *ek = s_e + lane + (ks << 2) * GEN_THREADS;
                s0 = fma(f01.x, ek[0], s0);
                s1 = fma(f01.y, ek[GEN_THREADS], s1);
                s0 = fma(f23.x, ek[2 * GEN_THREADS], s0);
                s1 = fma(f23.y, ek[3 * GEN_THREADS], s1);
            }
            s_dr[r][lane] = s0 + s1;
        }
        if (a.n_xo) {                                                     // trapezoid int_K at the new point (bq_c.pyx:585-593)
            double s0 = 0.0;
            for (int j = warp; j < a.n_xo; j += GEN_WARPS) s0 = fma(wp[j], kernel_exp(x - xo[j], nhl, kind, hp_l), s0);
            s_part[3][warp][lane] = s0;
        }
        __syncthreads();                                                  // every warp is done with the K_l vectors
        // ---- K_tl pass: tm = k_t . a_tl, qt = |L_tl^-1 k_t|^2
        double tmv = 0.0;
        for (int k = warp; k < ns; k += GEN_WARPS) {
            const double e = kernel_exp(x - xs[k], nhtl, kind, hp_tl);
            s_e[k * GEN_THREADS + lane] = e;
            tmv = fma(atl[k], e, tmv);
        }
        s_part[2][warp][lane] = tmv;
        __syncthreads();
        double qt = 0.0;
        for (int r = warp; r < ns; r += GEN_WARPS) {
            const double v = tri_row_dot(Ft, r, s_e, lane);
            qt = fma(v, v, qt);
        }
        s_part[1][warp][lane] = qt;
        __syncthreads();
        if (warp != 0) continue;                                          // (the loop is uniform: every warp comes back to the barrier)
        // warp 0: partial sums in warp order (deterministic)
        qs = qt = tmv = 0.0;
        double b_trap = 0.0;
        bool close = false;
#pragma unroll
        for (int w = 0; w < GEN_WARPS; ++w) {
            qs += s_part[0][w][lane]; qt += s_part[1][w][lane]; tmv += s_part[2][w][lane];
            if (a.n_xo) b_trap += s_part[3][w][lane];
            close |= s_close[w][lane] != 0;
        }
        // ---- tail (the branches of bq.py:447-527 / bq_c.pyx:425-490; same order of operations as bq_score.cu)
        double esm, em;
        int st = ST_OK;
        if (live) {
            if (!fin) {
                esm = em = nan("");
                st = ST_XA_BAD;
            } else if (close) {
                em = Zm; esm = Zm * Zm; st = ST_SHORTCUT;                 // bq.py:456-459
            } else {
                const double thresh = M[H_THRESH];
                unsigned mask = 0;
                for (int j = 0; j < nc; ++j) {
                    const double dc = xc[j] - x;
                    if (fabs(dc) < thresh) mask |= 1u << j;               // bq.py:470 (strict <)
                    s_dr[j][lane] = fma(c_l, kernel_exp(dc, nhl, kind, hp_l), s_dr[j][lane]);     // w = k_c + W k_s
                }
                double qc = 0, vg = 0, va = 0, bg = 0, kaa;
                bool pd = true;
                if (mask == 0) {
                    const double *Lc = M + lay.off_lcc0, *ug = M + lay.off_ug0, *ua = M + lay.off_ua0, *rd = M + lay.off_rd0;
                    for (int i = 0; i < nc; ++i) {
                        double s = s_dr[i][lane];
                        for (int k = 0; k < i; ++k) s = fma(-Lc[i * NC_MAX + k], s_dr[k][lane], s);
                        s *= rd[i];
                        s_dr[i][lane] = s;
                        qc = fma(s, s, qc); vg = fma(s, ug[i], vg); va = fma(s, ua[i], va);
                        bg = fma(ug[i], ua[i], bg);
                    }
                    kaa = M[H_KAA_E];
                } else {
                    // jitter on the close candidates (bq.py:471-473): refactorise the nc x nc Schur block
                    const double *S0 = M + lay.off_s0, *wb = M + lay.off_wb, *wa = M + lay.off_wa;
                    const double j1 = M[H_J1];
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
                            double s = s_dr[i][lane], sg = wb[i], sa = wa[i];
                            for (int k = 0; k < i; ++k) {
                                const double l = Lc[i * (i + 1) / 2 + k];
                                s -= l * s_dr[k][lane]; sg -= l * ug[k]; sa -= l * ua[k];
                            }
                            const double d = Lc[i * (i + 1) / 2 + i];
                            s /= d; sg /= d; sa /= d;
                            s_dr[i][lane] = s; ug[i] = sg; ua[i] = sa;
                            qc = fma(s, s, qc); vg = fma(s, sg, vg); va = fma(s, sa, va);
                            bg = fma(sg, sa, bg);
                        }
                    }
                    kaa = M[H_KAA_N];
                }
                const double s_ = kaa - (qs + qc);                        // Schur pivot of the new point
                if (!pd || !(s_ > 0.0)) {
                    em = Zm; esm = Zm * Zm; st = ST_NOTPD;                // bq.py:481-490
                } else {
                    const double ba = M[H_BA_S] + bg;                     // int_K(x_sc) . alpha_P
                    const double kg = s_dr[nc][lane] + vg;                // k_a . gamma_P
                    const double ka = s_dr[nc + 1][lane] + va;            // k_a . alpha_P
                    double b_a;
                    if (a.n_xo) {
                        b_a = c_l * b_trap;
                    } else {                                              // gauss_c.pyx:162: h^2 N(x_a | mu, w_l^2 + sigma^2)
                        const double diff = x - M[H_MU];
                        b_a = M[H_CB] * exp((diff * diff) * M[H_NHB]);
                    }
                    const double A_a = (b_a - kg) / s_;                   // bq_c.pyx:467-469
                    const double A_sc_l = ba - A_a * ka;                  // bq_c.pyx:470
                    const double tC = M[H_KTT] - qt;                      // gp_log_l.cov(x_a)            bq.py:496
                    const double a1 = tmv + 0.5 * tC;                     // int_exp_norm(1, tm, tC)      gauss_c.pyx:87
                    const double a2 = 2.0 * tmv + 2.0 * tC;               // int_exp_norm(2, tm, tC)
                    if (a1 > MAX_EXPONENT) {                              // bq_c.pyx:472-475
                        esm = em = INFINITY;
                    } else {
                        const double e1 = exp(a1);
                        em = A_sc_l + A_a * e1;                           // bq_c.pyx:477
                        if (a2 > MAX_EXPONENT) {
                            esm = INFINITY;                               // bq_c.pyx:479-483
                        } else {
                            const double e2 = exp(a2);
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
            if (epi) {
                const double evv = __dsub_rn(__dadd_rn(__dmul_rn(Zm, Zm), M[H_ZV]), esm);
                a.ev[po] = evv;
                if (evv < best_v || (evv == best_v && po < best_i)) { best_v = evv; best_i = po; }
            }
            if (o_em) o_em[po] = em;
            if (o_st) o_st[po] = st;
            if (st) {
                if (a.flags) atomicOr(a.flags + inst, st);
                cta_st |= st;
            }
        }
        __syncwarp();
    }
    if (warp != 0) return;
    if (a.cta_flags) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cta_st |= __shfl_xor_sync(0xffffffffu, cta_st, o);
        if (lane == 0) a.cta_flags[blockIdx.y * gridDim.x + blockIdx.x] = cta_st;
    }
    if (epi && a.part_val) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double v2 = __shfl_xor_sync(0xffffffffu, best_v, o);
            const long long i2 = __shfl_xor_sync(0xffffffffu, best_i, o);
            if (v2 < best_v || (v2 == best_v && i2 < best_i)) { best_v = v2; best_i = i2; }
        }
        if (lane == 0) { a.part_val[blockIdx.x] = best_v; a.part_idx[blockIdx.x] = best_i; }
    }
}

// Same contract as launch_score (bq_score.cu): grid_x receives the number of CTAs per instance (= partials of the fused
// epilogue).  Prediction mode is not offered by this kernel.
cudaError_t launch_score_generic(const ScoreArgs &a, int n_inst, cudaStream_t stream, int *grid_x) {
    if (a.predict) return cudaErrorNotSupported;
    if (a.na <= 0 || n_inst <= 0) { if (grid_x) *grid_x = 0; return cudaSuccess; }
    long long gx = ((long long)a.na + GEN_THREADS - 1) / GEN_THREADS;
    if (gx > GEN_MAX_GRID) gx = GEN_MAX_GRID;
    const size_t bytes = sizeof(double) * (size_t)a.lay.nsp_cap * GEN_THREADS;
    cudaError_t e = cudaFuncSetAttribute(bq_score_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return e;
    bq_score_generic_kernel<<<dim3((unsigned)gx, (unsigned)n_inst), GEN_THREADS * GEN_WARPS, bytes, stream>>>(a);
    if (grid_x) *grid_x = (int)gx;
    return cudaGetLastError();
}

}  // namespace bqb
