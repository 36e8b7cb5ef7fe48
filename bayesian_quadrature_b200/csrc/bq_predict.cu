// Prediction kernel: gp_l.mean(x) and diag gp_log_l.cov(x) (the two factors of BQ.l_mean / BQ.l_var, bq.py:177-231) for every
// kind of batch -- tensor-core or generic, Gaussian or periodic kernel, every capacity class, any s_l.
//
//   l_mean  = K_l(x, x_sc) alpha_l = c_l sum_k alpha_k e_l(x - x_sc[k])     alpha_l = (K_l + s_l^2 I)^-1 l_sc, stored by the
//                                                                             setup kernel (gp_l.inv_Kxx_y)
//   v_log_l = K_tl(x, x) - |L_tl^-1 k_tl(x)|^2                                 L_tl^-1 from the model block (c_tl-scaled
//                                                                             fragment-ordered copy, as the scoring kernels read it)
//
// The CTA shape of the generic scoring kernel (bq_score_generic.cu): eight warps share a tile of 32 query points, lane = point,
// plain FP64.  The warps split the terms of the mean and the rows of L_tl^-1; warp 0 adds the partial sums in warp order, so a
// point's result depends on nothing but its instance and its value (not on the other rows or points of the launch).  Unlike the
// scoring kernels' prediction mode there is no shortcut and no jitter pattern; a non-finite point gives NaN in both outputs.
// About half the work of a generic scoring pass: n + ns kernel evaluations and ns^2 / 2 FMAs per point.
#include "bq_common.cuh"

namespace bqb {

constexpr int PRED_MAX_GRID = 2048;          // CTAs per instance (grid-stride over the points beyond that)

__global__ void __launch_bounds__(GEN_THREADS * GEN_WARPS) bq_predict_kernel(PredictArgs a) {
    extern __shared__ double s_e[];                                  // [nsp][32] K_tl exponentials of the tile's points
    __shared__ double s_part[2][GEN_WARPS][GEN_THREADS];             // per-warp partial sums: mean, qt
    const Layout lay = a.lay;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int inst = a.rows ? a.rows[a.row0 + blockIdx.y] : a.row0 + blockIdx.y;
    const double *M = a.models + (size_t)inst * lay.total;
    const int ns = (int)M[H_NS], nc = (int)M[H_NC], nsp = (int)M[H_NSP];
    const int n = ns + nc;
    const int kind = (int)M[H_KIND];
    const double hp_tl = M[H_HP_TL], hp_l = M[H_HP_L];
    const double c_l = M[H_CL], nhl = M[H_NHL], nhtl = M[H_NHTL], ktt = M[H_KTT];
    const double *xs = M + lay.off_xs, *xc = M + lay.off_xc, *Ft = M + lay.off_af_tl_tri;
    const double *al = a.alpha + (size_t)inst * a.alpha_stride;
    const double *xq = a.x + (size_t)inst * a.x_stride;
    double *o_m = a.l_mean + (size_t)inst * a.out_stride;
    double *o_v = a.v_log_l + (size_t)inst * a.out_stride;

    if (warp == 0)
        for (int k = ns; k < nsp; ++k) s_e[k * GEN_THREADS + lane] = 0.0;  // padding of the last k-step
    for (long long t0 = (long long)blockIdx.x * GEN_THREADS; t0 < a.na; t0 += (long long)gridDim.x * GEN_THREADS) {
        const long long p = t0 + lane;
        const bool live = p < a.na;
        const double xv = live ? xq[p] : 0.0;
        const bool fin = live && isfinite(xv);
        const double x = fin ? xv : 0.0;
        __syncthreads();                                                  // the previous tile's tail has left s_part / s_e
        // ---- mean: sum_k alpha_k e_l(x - x_sc[k]) over the observations and the candidates (model order)
        double m = 0.0;
        for (int k = warp; k < n; k += GEN_WARPS) {
            const double xk = k < ns ? xs[k] : xc[k - ns];
            m = fma(al[k], kernel_exp(x - xk, nhl, kind, hp_l), m);
        }
        s_part[0][warp][lane] = m;
        // ---- variance: e[k] = exp part of K_tl(x, x_s[k]);  qt = |(c_tl L_tl^-1) e|^2
        for (int k = warp; k < ns; k += GEN_WARPS) s_e[k * GEN_THREADS + lane] = kernel_exp(x - xs[k], nhtl, kind, hp_tl);
        __syncthreads();
        double qt = 0.0;
        for (int r = warp; r < ns; r += GEN_WARPS) {
            const double v = tri_row_dot(Ft, r, s_e, lane);
            qt = fma(v, v, qt);
        }
        s_part[1][warp][lane] = qt;
        __syncthreads();
        if (warp != 0 || !live) continue;                                 // (every warp comes back to the barrier)
        m = qt = 0.0;
#pragma unroll
        for (int w = 0; w < GEN_WARPS; ++w) { m += s_part[0][w][lane]; qt += s_part[1][w][lane]; }
        o_m[p] = fin ? c_l * m : nan("");
        o_v[p] = fin ? ktt - qt : nan("");
    }
}

// Instances rows[row0 .. row0 + n_rows) (rows null: row0 .. row0 + n_rows), at most 65535 of them (gridDim.y)
cudaError_t launch_predict(const PredictArgs &a, int n_rows, cudaStream_t stream) {
    if (a.na <= 0 || n_rows <= 0) return cudaSuccess;
    long long gx = ((long long)a.na + GEN_THREADS - 1) / GEN_THREADS;
    if (gx > PRED_MAX_GRID) gx = PRED_MAX_GRID;
    const size_t bytes = sizeof(double) * (size_t)a.lay.nsp_cap * GEN_THREADS;
    cudaError_t e = cudaFuncSetAttribute(bq_predict_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return e;
    bq_predict_kernel<<<dim3((unsigned)gx, (unsigned)n_rows), GEN_THREADS * GEN_WARPS, bytes, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace bqb
