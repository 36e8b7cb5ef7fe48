// Shared definitions of the B200 expected-variance scoring path: the device-resident model
// block layout, status bits, the FP64 DMMA wrapper and the table-driven exp used to generate
// cross-kernel fragments.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

namespace bqb {

// ---- per-point status bits (mirror the reference's branches; host turns them into exceptions)
constexpr int ST_OK = 0;
constexpr int ST_SHORTCUT = 1;   // bq.py:456-459   x_a isclose to an observation -> (Zm^2, Zm)
constexpr int ST_NOTPD = 2;      // bq.py:481-490   bordered matrix not PD      -> (Zm^2, Zm)
constexpr int ST_ESM_INF = 4;    // bq.py:522-523   logger.warn
constexpr int ST_EM_INF = 8;     // bq.py:524-525   logger.warn
constexpr int ST_ESM_BAD = 16;   // bq.py:514-517   RuntimeError (NaN or negative esm)
constexpr int ST_EM_BAD = 32;    // bq.py:518-520   RuntimeError (NaN em)
constexpr int ST_XA_BAD = 64;    // bq.py:451-452   ValueError (NaN / inf x_a)

// ---- setup status (per model instance)
constexpr int SETUP_OK = 0;
constexpr int SETUP_KTL_NOTPD = 1;    // gp_log_l.Kxx not positive definite
constexpr int SETUP_KL_NOTPD = 2;     // gp_l.Kxx not positive definite
constexpr int SETUP_MEAN_TOO_LARGE = 3;  // bq.py:945-947 "GP mean is too large"
constexpr int SETUP_BAD_INPUT = 4;    // non-finite / non-positive inputs

constexpr int NC_MAX = 16;            // candidates per instance supported on device
constexpr int EXP_TAB_MAX = 2048;     // device table: [0, 2048) = 2^(j/2048), [2048, 2560) = 2^(j/512)
constexpr double MAX_EXPONENT = 707.0101241711442;   // log(2^1020): gauss_c.pyx:16, bq.py:16
constexpr double EPS = 2.220446049250313e-16;        // np.finfo(float64).eps, bq_c.pyx:28

// ---- header slots of a model block (doubles)
enum Hdr {
    H_NS = 0, H_NC, H_NSP, H_STATUS, H_CL, H_NHL, H_CTL, H_NHTL, H_KAA_E, H_KAA_N, H_J1, H_KTT, H_MU,
    H_CB, H_NHB, H_ZM, H_ZV, H_THRESH, H_LOGLH, H_BA_S, H_NDB, H_WL, H_TOL2MAX,
    H_KIND, H_HP_TL, H_HP_L,          // kernel kind (0 Gaussian, 1 periodic) and 1 / (2 p) of the two kernels (generic path)
    H_COUNT = 32
};

// Model block layout (offsets in doubles) for an instance capacity of nsp_cap observations
// (multiple of 8) and NC_MAX candidates.  Every array is padded so that padded observations
// contribute exactly zero.
struct Layout {
    int nsp_cap;     // padded observation capacity (multiple of 8)
    int nb_cap;      // row blocks of 8
    int nks_cap;     // k-steps of 4
    int off_xs, off_tol, off_atl, off_xc, off_lc, off_s0, off_lcc0, off_wb, off_wa, off_ug0, off_ua0, off_rd0;
    int off_af_l_tri, off_af_l_dense, off_af_tl_tri;
    int n_small;     // doubles before the fragment arrays (header + vectors + small matrices)
    int total;       // doubles per instance (multiple of 32)
};

__host__ __device__ inline int tri_frags(int nb) { return nb * (nb + 1); }   // sum_{rb<nb} (2 rb + 2)

__host__ __device__ inline Layout make_layout(int nsp_cap) {
    Layout L;
    L.nsp_cap = nsp_cap;
    L.nb_cap = nsp_cap / 8;
    L.nks_cap = nsp_cap / 4;
    int o = H_COUNT;
    L.off_xs = o; o += nsp_cap;
    L.off_tol = o; o += nsp_cap;
    L.off_atl = o; o += nsp_cap;
    L.off_xc = o; o += NC_MAX;
    L.off_lc = o; o += NC_MAX;
    L.off_s0 = o; o += NC_MAX * NC_MAX;
    L.off_lcc0 = o; o += NC_MAX * NC_MAX;
    L.off_wb = o; o += NC_MAX;
    L.off_wa = o; o += NC_MAX;
    L.off_ug0 = o; o += NC_MAX;
    L.off_ua0 = o; o += NC_MAX;
    L.off_rd0 = o; o += NC_MAX;                         // 1 / diag(L_cc)
    o = (o + 31) & ~31;
    L.n_small = o;
    L.off_af_l_tri = o; o += tri_frags(L.nb_cap) * 32;
    L.off_af_l_dense = o; o += 3 * L.nks_cap * 32;      // up to 3 dense row blocks (nc + 2 <= 24 rows)
    L.off_af_tl_tri = o; o += tri_frags(L.nb_cap) * 32;
    L.total = o;
    return L;
}

// Arguments of one scoring launch (bq_score.cu); shared with the C-ABI layer (bq_capi.cu)
struct ScoreArgs {
    const double *models = nullptr;     // [B][lay.total]
    Layout lay;
    const double *x_a = nullptr;        // [na] (xa_stride = 0) or [B / xa_group][xa_stride]
    long long xa_stride = 0;
    int xa_group = 1;                   // instance inst reads query row inst / xa_group (samples of one problem share a grid)
    int na = 0;
    double *esm = nullptr, *em = nullptr;   // [B][out_stride]; em may be null (esm too when ev is given)
    int *status = nullptr;              // [B][out_stride]; may be null
    long long out_stride = 0;
    const double *exp_tab = nullptr;    // [EXP_TAB]
    int *flags = nullptr;               // [B] OR of every point's status bits (may be null)
    int *cta_flags = nullptr;           // [gridDim.y][gridDim.x] the same per CTA, written with plain stores (may be null)
    int inst0 = 0;
    int ndb_max = 1;                    // dense row blocks to reserve scratch for: ceil((max nc + 2) / 8)
    // optional fused epilogue of choose_next / expected_Z_var (single-instance launches only):
    double *ev = nullptr;               // [na] expected variance Zm^2 + Zv - esm (bq.py:374-377); may be null
    double *part_val = nullptr;         // [gridDim.x] per-CTA minimum of ev ...
    long long *part_idx = nullptr;      // ... and the first index attaining it (np.argmin semantics); may be null
    int chunk_frags = 0;                // streamed kernels: fragments per operand chunk (set by launch_score)
    int nb_max = 0, nrow_max = 0;       // largest row-block count / nc + 2 over the batch's instances (0: unknown -> class maximum)
    int nb_res = 0, nrow_res = 0;       // what the launch sizes its shared memory for (set by launch_score from the two above)
    const int *perm = nullptr;          // x_a is sorted: perm[p] = position of point p in the caller's vector (outputs go there)
    int predict = 0;                    // 1: prediction mode (esm <- gp_l.mean(x), em <- diag gp_log_l.cov(x))
    double cut_arg = 72.0;              // relevance cut-off of a cross-kernel exponent below its point's largest (+inf: dense)
    int force_wide = 0;                 // band-relative kernels: every warp takes the wide (windowed) path (tests)
    unsigned long long *work = nullptr; // optional counter: DMMA instructions executed (all warps, atomically added)
    // generic path (bq_score_generic.cu): non-Gaussian kernels and / or the trapezoid approximation of int_K
    const double *xo = nullptr;         // [n_xo] approximation grid (shared) or [B][xo_stride]
    const double *wp = nullptr;         // [B][n_xo] trapezoid weight x prior density, written by the setup kernel
    int n_xo = 0;                       // 0: closed-form int_K (Gaussian kernel)
    long long xo_stride = 0;
};

// Arguments of one setup launch (bq_setup2.cu); shared with the C-ABI layer (bq_capi.cu)
struct SetupArgs {
    // inputs, one row per instance
    const int *ns, *nc;
    const double *x_s, *l_s;   // [B][in_stride]
    const double *x_c;         // [B][NC_MAX]
    const double *hyp;         // [B][6]  h_tl, w_tl, s_tl, h_l, w_l, s_l
    const double *prior;       // [B][3]  mu, sigma2, candidate_thresh
    int in_stride;
    int check_max;             // apply the bq.py:942-947 guard
    // outputs
    double *models;            // [B][lay.total]
    Layout lay;
    // scratch, per instance: the packed triangle of instances too large for shared memory (setup2_scratch_stride)
    double *work;
    size_t work_stride;
    int inst0;                 // first instance of this chunk
    const int *inst_list;      // bq_setup2.cu: when set, CTA b works on instance inst_list[inst0 + b] (launch groups by size)
    int n_max, nc_max;         // bq_setup2.cu: largest ns + nc / nc over the instances of the launch (size the shared memory)
    // non-Gaussian kernels / trapezoid approximation (bq_c.pyx:216-261, :358-422, :538-598); bq_setup2.cu only
    int kind;                  // 0: gp.GaussianKernel, 1: gp.PeriodicKernel
    const double *period;      // [B][2] p of gp_log_l's and gp_l's kernel (kind 1), else null
    const double *xo, *pxo;    // approximation grid and prior density on it: [n_xo] (xo_stride = 0) or [B][xo_stride]
    int n_xo;                  // 0: closed-form integrals
    long long xo_stride;
    double *wp;                // out [B][n_xo]: trapezoid weight x prior density
    double *gz;                // scratch [launch instances][n_xo]
    // out [B][alpha_stride]: alpha_l = (K_l + s_l^2 I)^-1 l_sc (gp_l.inv_Kxx_y) in model order, zero padded (may be null;
    // last members: the other parameters keep their offsets)
    double *alpha;
    long long alpha_stride;
};

// Arguments of one launch of the prediction kernel (bq_predict.cu); shared with the C-ABI layer (bq_capi.cu)
struct PredictArgs {
    const double *models = nullptr;     // [n_inst][lay.total]
    Layout lay;
    const double *alpha = nullptr;      // [n_inst][alpha_stride], written by the setup kernel
    long long alpha_stride = 0;
    const int *rows = nullptr;          // CTA row y works on instance rows[row0 + y] (null: instance row0 + y)
    int row0 = 0;
    const double *x = nullptr;          // [na] (x_stride = 0) or [n_inst][x_stride]
    long long x_stride = 0;
    int na = 0;
    double *l_mean = nullptr, *v_log_l = nullptr;   // [n_inst][out_stride]
    long long out_stride = 0;
};

// Arguments of one launch of the log-likelihood gradient kernel (bq_setup2.cu); shared with the C-ABI layer (bq_capi.cu).
// It reads the staged inputs of a batch and writes nothing but `out`.
constexpr int LLG_OUT = 8;     // doubles per output row: log_lh, d/d(h_tl, w_tl, s_tl, h_l, w_l, s_l), status
constexpr int LLG_OUT_PERIODIC = 10;   // periodic kernel: log_lh, d/d(h_tl, w_tl, s_tl, h_l, w_l, s_l, p_tl, p_l), status
struct LLGradArgs {
    const int *ns, *nc;
    const double *x_s, *l_s;   // [n_inst][in_stride] (in_stride = the batch's observation capacity)
    const double *x_c;         // [n_inst][NC_MAX]
    int in_stride;
    const double *hyp;         // [n_eval][6]  h_tl, w_tl, s_tl, h_l, w_l, s_l of each row
    const int *inst;           // [n_eval] instance of each row (null: row e is instance e)
    int e0;                    // first row of this launch
    int check_max;             // apply the bq.py:942-947 guard
    int n_max, nc_max;         // largest ns + nc / nc over the batch's instances (size the shared memory)
    double *work;              // scratch per CTA for instances too large for shared memory (setup2_scratch_stride)
    size_t work_stride;
    double *out;               // [n_eval][LLG_OUT], periodic kernel [n_eval][LLG_OUT_PERIODIC]
    const double *period;      // periodic kernel: [n_eval][2] p of gp_log_l's and gp_l's kernel of each row (last member:
                               // the Gaussian instantiations keep their parameter offsets)
};

#ifdef __CUDACC__

// D(8x8) += A(8x4) * B(4x8), FP64 tensor path (SASS: DMMA.8x8x4).  Lane l holds
// A[l>>2][l&3], B[l&3][l>>2], C/D[l>>2][2*(l&3) + {0,1}].
__device__ __forceinline__ void dmma(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// ---- table-driven FP64 exp.  T[j] = 2^(j/N) lives in shared memory (N = 2048 or 512).
//
// DMMA and DFMA share one FP64 datapath on B200 (profiles/fp64_mix_r01.json), so every FP64 instruction
// spent on the cross-kernel exponentials is taken from the GEMM.  libm's exp costs ~21 FP64-pipe
// operations; exp_kernel below costs 7 (N = 2048) or 8 (N = 512).
template <int N> struct ExpC;
template <> struct ExpC<2048> {
    static constexpr int SHIFT = 11;
    static constexpr double INVN = 0x1.71547652b82fep+11;          // N / ln 2
    static constexpr double HI = 0x1.62e42fec00000p-12;            // ln2 / N, top 31 bits
    static constexpr double LO = 0x1.d1cf79abc9e3bp-43;
    static constexpr double MAGIC_B = 6755399443150848.0;          // 1.5 * 2^52 + 1023 * N
};
template <> struct ExpC<512> {
    static constexpr int SHIFT = 9;
    static constexpr double INVN = 0x1.71547652b82fep+9;
    static constexpr double HI = 0x1.62e42fef00000p-10;            // top 33 bits
    static constexpr double LO = 0x1.473de6af278edp-43;
    static constexpr double MAGIC_B = 6755399441579520.0;          // 1.5 * 2^52 + 1023 * N
};
constexpr double EXP_MAGIC = 6755399441055744.0;                   // 1.5 * 2^52

// exp(d2 * nh) for d2 >= 0, nh < 0, given C = nh * N / ln 2 (rounded once).  The argument is reduced in
// *table units*: u = d2 * C, k = rint(u), r = u - k computed by ONE fma (exact product, |r| <= 1/2), so no
// hi/lo split of ln 2 is needed; exp(r ln2 / N) - 1 is a degree-3 (N = 2048, fitted, 0.05 ulp) or degree-4
// (N = 512, Taylor, 0.01 ulp) polynomial in r.  Total error ~1 ulp + |arg| * 1.6e-16 (the rounding of d2
// and of C, i.e. a 1e-16 relative perturbation of the length scale w).
// d2 is clamped to d2max (<= 700 / |nh|) with ONE integer min on its high word (non-negative doubles order
// like their bit patterns), so far-away points give ~1e-304 instead of an exact 0 and the result is always a
// normal number; it also maps d2 = +inf to a finite value.  All of this keeps work off the FP64 pipe, which a
// warp instruction occupies for 2 issue cycles (DSETP / DMNMX would cost as much as a DFMA).
// The exp phase is issue bound (ncu: 9 FP64 + 11 other instructions per element), so the integer side is kept
// minimal: the rounding constant carries the exponent bias (k + 1023 N in the low word of t), hence the scale
// 2^(k >> log2 N) is merged into the table value by ONE shift and ONE bit-select (LOP3) *before* the final FMAs
// -- no mask, no add, and nothing integer at the end of the dependency chain.
template <int N>
__device__ __forceinline__ double exp_kernel(double d2, double C, int d2max_hi, const double *__restrict__ tab) {
    d2 = __hiloint2double(min(__double2hiint(d2), d2max_hi), __double2loint(d2));
    const double t = fma(d2, C, ExpC<N>::MAGIC_B);
    const int ki = __double2loint(t);                      // round(u) + 1023 N  (> 0: the clamp keeps u >= -1010 N)
    const double kf = t - ExpC<N>::MAGIC_B;
    const double r = fma(d2, C, -kf);
    double q;
    if (N == 2048) {
        q = fma(0x1.c6b08d79d8fa9p-38, r, 0x1.ebfbe00896926p-25);
        q = fma(q, r, 0x1.62e42fefa39efp-12);
    } else {
        q = fma(0x1.3b2ab6fba4e77p-43, r, 0x1.c6b08d704a0c0p-32);
        q = fma(q, r, 0x1.ebfbdff82c58fp-21);
        q = fma(q, r, 0x1.62e42fefa39efp-10);
    }
    const double T = tab[ki & (N - 1)];                    // in [1, 2): exponent field 0x3ff, replaced below
    // biased exponent (ki >> log2 N) into bits 20..30, mantissa bits of T kept: (T_hi & 0xfffff) | ((ki << s) & ~0xfffff)
    int hs;                                                // bit-select: one LOP3 (the compiler emits two for the C form)
    asm("lop3.b32 %0, %1, %2, 0x000fffff, 0xE4;" : "=r"(hs) : "r"(__double2hiint(T)), "r"(ki << (20 - ExpC<N>::SHIFT)));
    const double Ts = __hiloint2double(hs, __double2loint(T));
    return fma(Ts * r, q, Ts);
}

// high word of the largest d2 the kernel exponent may see: 700 / |nh| (exp(-700) ~ 1e-304)
__device__ __forceinline__ int exp_d2max_hi(double nh) { return __double2hiint(700.0 / fabs(nh)); }

// exp(x) for any finite x <= 709 (used a few times per point in the tail, where the argument can be large
// and positive): classic Cody-Waite reduction with a hi/lo split of ln2/N so that large |x| keeps full
// relative accuracy; Taylor degree 3 (N = 2048, 0.31 ulp) or 4 (N = 512).
template <int N>
__device__ __forceinline__ double exp_tab(double x, const double *__restrict__ tab) {
    const double t = fma(x, ExpC<N>::INVN, EXP_MAGIC);
    const int ki = __double2loint(t);
    const double kf = t - EXP_MAGIC;
    double r = fma(kf, -ExpC<N>::HI, x);
    r = fma(kf, -ExpC<N>::LO, r);
    double q = (N == 2048) ? fma(r, 1.0 / 6.0, 0.5) : fma(fma(r, 1.0 / 24.0, 1.0 / 6.0), r, 0.5);
    const double p = fma(q, r * r, r);
    const double T = tab[ki & (N - 1)];
    double y = fma(T, p, T);
    y = __hiloint2double(__double2hiint(y) + ((ki >> ExpC<N>::SHIFT) << 20), __double2loint(y));
    return (x < -708.0) ? 0.0 : y;
}

// exponent part of a stationary kernel at distance d: Gaussian exp(nh d^2) (nh = -1 / (2 w^2)); gp.PeriodicKernel
// h^2 exp(-2 sin^2(d / (2 p)) / w^2) = h^2 exp(nh D^2) with the chordal distance D = 2 sin(d hp), hp = 1 / (2 p)
__device__ __forceinline__ double kernel_exp(double d, double nh, int kind, double hp) {
    if (kind) d = 2.0 * sin(d * hp);
    return exp((d * d) * nh);
}

// ---- plain-FP64 kernels (bq_score_generic.cu, bq_predict.cu): eight warps share a tile of 32 query points, lane = point
constexpr int GEN_THREADS = 32;              // points per tile (= lanes)
constexpr int GEN_WARPS = 8;                 // warps of a CTA: they share the tile

// sum_{k <= r} F[r][k] e[k] for row r of a triangular fragment-ordered operand: a k-step is four consecutive doubles of the
// row (32-byte aligned: two 16-byte warp-uniform loads); entries with k > r are stored as zeros, so whole k-steps are used
// (the e buffer, [k][lane] in shared memory, is zero for k >= ns)
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

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

#endif  // __CUDACC__

}  // namespace bqb
