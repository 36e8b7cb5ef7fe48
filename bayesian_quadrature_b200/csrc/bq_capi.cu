// C-ABI of the B200 expected-variance scoring library (declared in include/bq_b200.h).
// Plain pointers and sizes only; no torch types.  Every entry point returns 0 on success,
// a negative BQB_E* code for argument errors and a positive cudaError_t otherwise; the
// message is kept per thread (bqb_last_error).
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/bq_b200.h"
#include "bq_common.cuh"

namespace bqb {
cudaError_t launch_setup2(const SetupArgs &a, int n_inst, cudaStream_t stream);
cudaError_t launch_llgrad(LLGradArgs a, int n_rows, int work_inst, cudaStream_t stream, int *launches, int kind);
int setup2_two_cta_limit(int nc_max);
size_t setup2_scratch_stride(int cap);
cudaError_t launch_score(const ScoreArgs &a, int n_inst, int sm_count, cudaStream_t stream, int *grid_x = nullptr);
cudaError_t launch_score_generic(const ScoreArgs &a, int n_inst, cudaStream_t stream, int *grid_x);
cudaError_t launch_predict(const PredictArgs &a, int n_rows, cudaStream_t stream);
cudaError_t launch_argmin_partials(double *bv, long long *bi, int nblocks, long long offset, double *pair, cudaStream_t s);
cudaError_t launch_pack_info(const double *models, long long model_stride, int off_lc, int n_inst, double *out, cudaStream_t s);
cudaError_t launch_sum_neg_groups(const double *esm, long long stride, int n_groups, int group_size, long long na, double *acc,
                                  long long acc_stride, bool mean, cudaStream_t s);
cudaError_t launch_expected_var_rows(const double *models, long long model_stride, int inst0, int n_rows, const double *esm,
                                     long long esm_stride, long long na, double *out, long long out_stride, cudaStream_t s);
cudaError_t launch_argmin(const double *v, long long n, double *bv, long long *bi, int sm_count, long long offset, double *pair,
                          cudaStream_t s);
cudaError_t launch_argmin_rows(const double *v, long long stride, long long n, int rows, double *mins, long long *idxs,
                               cudaStream_t s);
cudaError_t launch_argmin_ties_rows(const double *v, long long stride, long long n, int rows, const double *mins, const double *u,
                                    long long *idxs, long long *counts, cudaStream_t s);
cudaError_t launch_argmin_exchange(const double *bv, const long long *bi, int nblocks, long long offset, long long cyc_block,
                                   void *const *peer_slots, int world, int rank, unsigned long long seq, double *out, cudaStream_t s);
cudaError_t sort_points(const double *d_x, int n, double *d_x_sorted, int *d_iota, int *d_perm, void *temp, size_t *temp_bytes,
                        cudaStream_t s);
cudaError_t launch_mt_seed(const unsigned *seeds, unsigned *mt, int *mti, int P, cudaStream_t s);
cudaError_t launch_add_observations(double *x_s, double *l_s, int *ns, int stride, const double *prior, const double *x_new,
                                    const double *l_new, int P, int *overflow, cudaStream_t s);
cudaError_t launch_draw_candidates(const double *x_s, const int *ns, int stride, const double *hyp, const double *prior,
                                   unsigned *mt, int *mti, int n_candidate, double *x_c, int *nc, int P, cudaStream_t s);
cudaError_t launch_draw_candidates_wrapped(const double *x_s, const int *ns, int stride, const double *period, const double *prior,
                                           unsigned *mt, int *mti, int n_candidate, double *x_c, int *nc, int P, cudaStream_t s);
}  // namespace bqb

using namespace bqb;

static thread_local std::string g_err;
static int fail(int code, const std::string &msg) { g_err = msg; return code; }
#define CU(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return fail((int)e_, std::string(#x) + ": " + cudaGetErrorString(e_)); } while (0)

struct bqb_batch {
    int device, n_inst, ns_cap, sm_count;
    Layout lay;
    double *d_models = nullptr, *d_tab = nullptr, *d_work = nullptr;
    int work_inst = 0;
    size_t work_stride = 0;
    // staged inputs: x_s / l_s rows have the device stride ns_cap, so that observations can be appended in place
    int *d_ns = nullptr, *d_nc = nullptr;
    bool staged = false;
    // device-resident active sampling (bq_round.cu)
    unsigned *d_mt = nullptr;          // [624][n_inst] Mersenne-Twister words
    int *d_mti = nullptr, *d_overflow = nullptr;
    std::vector<int> h_ns, h_nc;
    bool counts_fresh = false;         // h_ns / h_nc mirror d_ns / d_nc
    // non-Gaussian kernels / trapezoid approximation (bqb_batch_set_approx): generic scoring kernel
    int kind = 0, n_xo = 0;
    long long xo_stride = 0;
    bool generic = false;
    bool big_class = false;            // capacity 512: no tensor-core scoring kernels
    double *d_period = nullptr, *d_xo = nullptr, *d_pxo = nullptr, *d_wp = nullptr, *d_gz = nullptr;
    int *d_inst_list = nullptr;        // setup launch groups (instances ordered by size class)
    // alpha_l of every instance, written by each setup ([n_inst][alpha_stride], model order, zero padded), and the instance
    // list of bqb_predict_rows_device (grown on demand)
    double *d_alpha = nullptr;
    long long alpha_stride = 0;
    int *d_rows = nullptr;
    size_t cap_rows = 0;
    // bqb_batch_log_lh_grad(_periodic): hyper-parameter rows, periods, instance list and output rows (grown on demand)
    double *d_llg_hyp = nullptr, *d_llg_out = nullptr, *d_llg_period = nullptr;
    int *d_llg_inst = nullptr;
    size_t cap_llg = 0;
    // scoring: relevance cut-off (bq_score.cu, CUT_ARG; +inf = dense) and the optional executed-work counter
    double cut_arg = 72.0;
    unsigned long long *d_work_ctr = nullptr;
    // pre-sort of query vectors that do not look sorted (bq_sort.cu): 0 never, 1 automatic (default), 2 always
    int presort = 1;
    // host entry points with page-locked buffers: 1 = the kernel reads / writes them in place (zero copy, default), 0 = staged copies
    int zero_copy = 1;
    double *d_xsorted = nullptr;
    int *d_perm = nullptr, *d_iota = nullptr;
    void *d_sort_tmp = nullptr;
    size_t cap_sort = 0, cap_sort_tmp = 0;
    double *d_xs = nullptr, *d_ls = nullptr, *d_xc = nullptr, *d_hyp = nullptr, *d_prior = nullptr;
    // host-buffer scoring staging (grown on demand)
    double *d_xa = nullptr, *d_esm = nullptr, *d_em = nullptr;
    int *d_st = nullptr;
    size_t cap_xa = 0, cap_out = 0;
    int *d_flags = nullptr;
    cudaStream_t pipe[2] = {nullptr, nullptr};
    int *h_flags = nullptr;            // pinned
    int *h_cta_flags = nullptr;        // pinned, mapped: per-CTA status words of the zero-copy scoring launch
    double *d_red_val = nullptr;
    long long *d_red_idx = nullptr;
    std::vector<double> h_hdr, h_lc;   // per-instance headers and l_c rows fetched by the last setup
    double *d_info = nullptr, *h_info = nullptr;       // [n_inst][H_COUNT + NC_MAX] packed on the device / page-locked mirror
    bool ready = false;
    int ndb_max = 1;
    int nb_max = 0, nrow_max = 0;      // largest ceil(ns / 8) and nc + 2 over the instances (sizes the kernels' shared memory)
    unsigned long long launches = 0;
};

extern "C" {

const char *bqb_last_error(void) { return g_err.c_str(); }

int bqb_version(void) { return 100; }

int bqb_device_count(int *count) {
    CU(cudaGetDeviceCount(count));
    return 0;
}

int bqb_ns_capacity(int ns) {
    if (ns < 1) return BQB_EINVAL;
    if (ns <= 16) return 16;
    if (ns <= 64) return 64;
    if (ns <= 128) return 128;
    if (ns <= 160) return 160;
    if (ns <= 256) return 256;
    if (ns <= 512) return 512;          // generic (plain FP64) scoring kernel only: the tensor-core kernels' k-step masks end at 256
    return BQB_EUNSUPPORTED;
}

int bqb_batch_create(bqb_batch **out, int device, int n_inst, int ns_max) {
    if (!out || n_inst < 1) return fail(BQB_EINVAL, "bqb_batch_create: bad arguments");
    const int cap = bqb_ns_capacity(ns_max);
    if (cap < 0) return fail(cap, "bqb_batch_create: ns_max outside the supported range [1, 512]");
    CU(cudaSetDevice(device));
    bqb_batch *b = new bqb_batch();
    b->device = device; b->n_inst = n_inst; b->ns_cap = cap; b->lay = make_layout(cap);
    // (two attribute queries, not cudaGetDeviceProperties: that call alone took 15-20 ms per batch on this pool's hosts,
    // more than everything else a hyper-parameter batch of choose_next does)
    int cc_major = 0, sm_count = 0;
    CU(cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, device));
    CU(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, device));
    if (cc_major < 10) { delete b; return fail(BQB_EUNSUPPORTED, "bqb_batch_create: needs an sm_100a device (B200)"); }
    b->sm_count = sm_count;
    CU(cudaMalloc(&b->d_models, sizeof(double) * (size_t)n_inst * b->lay.total));
    CU(cudaMalloc(&b->d_tab, sizeof(double) * (2048 + 512)));
    std::vector<double> tab(2048 + 512);
    for (int j = 0; j < 2048; ++j) tab[j] = (double)exp2l((long double)j / 2048);
    for (int j = 0; j < 512; ++j) tab[2048 + j] = (double)exp2l((long double)j / 512);
    CU(cudaMemcpy(b->d_tab, tab.data(), sizeof(double) * tab.size(), cudaMemcpyHostToDevice));
    b->work_inst = n_inst < 2048 ? n_inst : 2048;
    if (cap > 256) {
        // 257 .. 512 observations: generic scoring
        b->big_class = true;
        b->generic = true;
        if (b->work_inst > 256) b->work_inst = 256;
    }
    // setup scratch sized for the capacity CLASS, because bqb_batch_stage and bqb_batch_add_observations let ns grow up
    // to bqb_batch_capacity(), not just up to ns_max
    b->work_stride = setup2_scratch_stride(cap);
    if (b->work_stride) CU(cudaMalloc(&b->d_work, sizeof(double) * b->work_stride * b->work_inst));
    CU(cudaMalloc(&b->d_ns, sizeof(int) * n_inst));
    CU(cudaMalloc(&b->d_nc, sizeof(int) * n_inst));
    CU(cudaMalloc(&b->d_xs, sizeof(double) * (size_t)n_inst * cap));
    CU(cudaMalloc(&b->d_ls, sizeof(double) * (size_t)n_inst * cap));
    CU(cudaMalloc(&b->d_xc, sizeof(double) * (size_t)n_inst * NC_MAX));
    CU(cudaMalloc(&b->d_hyp, sizeof(double) * (size_t)n_inst * 6));
    CU(cudaMalloc(&b->d_prior, sizeof(double) * (size_t)n_inst * 3));
    b->alpha_stride = cap + NC_MAX;
    CU(cudaMalloc(&b->d_alpha, sizeof(double) * (size_t)n_inst * b->alpha_stride));
    CU(cudaMalloc(&b->d_red_val, sizeof(double) * 4096));
    CU(cudaMalloc(&b->d_red_idx, sizeof(long long) * 4096));
    if (getenv("BQB_DENSE") && atoi(getenv("BQB_DENSE"))) b->cut_arg = INFINITY;
    b->h_hdr.resize((size_t)n_inst * H_COUNT);
    b->h_lc.resize((size_t)n_inst * NC_MAX);
    CU(cudaMalloc(&b->d_info, sizeof(double) * (size_t)n_inst * (H_COUNT + NC_MAX)));
    CU(cudaMallocHost(&b->h_info, sizeof(double) * (size_t)n_inst * (H_COUNT + NC_MAX)));
    b->h_ns.resize(n_inst);
    b->h_nc.resize(n_inst);
    *out = b;
    return 0;
}

void bqb_batch_destroy(bqb_batch *b) {
    if (!b) return;
    cudaSetDevice(b->device);
    void *ptrs[] = {b->d_models, b->d_tab, b->d_work, b->d_ns, b->d_nc, b->d_xs, b->d_ls, b->d_xc, b->d_hyp, b->d_prior,
                    b->d_xa, b->d_esm, b->d_em, b->d_st, b->d_red_val, b->d_red_idx, b->d_flags, b->d_mt, b->d_mti, b->d_overflow, b->d_work_ctr, b->d_xsorted, b->d_perm, b->d_iota, b->d_sort_tmp,
                    b->d_period, b->d_xo, b->d_pxo, b->d_wp, b->d_gz, b->d_inst_list, b->d_llg_hyp, b->d_llg_out, b->d_llg_inst,
                    b->d_llg_period, b->d_alpha, b->d_rows};
    for (void *p : ptrs) if (p) cudaFree(p);
    for (cudaStream_t st : b->pipe) if (st) cudaStreamDestroy(st);
    if (b->h_flags) cudaFreeHost(b->h_flags);
    if (b->h_cta_flags) cudaFreeHost(b->h_cta_flags);
    if (b->d_info) cudaFree(b->d_info);
    if (b->h_info) cudaFreeHost(b->h_info);
    delete b;
}

// Largest ns + nc and nc over the staged instances (they size the shared memory of the setup and gradient kernels).
// The counts are fetched first when the device-side round kernels (add_observations, draw_candidates) changed them
// without the host seeing it.
static int staged_sizes(bqb_batch *b, cudaStream_t s, int *n_max_out, int *nc_max_out) {
    const int B = b->n_inst;
    if (!b->counts_fresh) {
        CU(cudaMemcpyAsync(b->h_ns.data(), b->d_ns, sizeof(int) * B, cudaMemcpyDeviceToHost, s));
        CU(cudaMemcpyAsync(b->h_nc.data(), b->d_nc, sizeof(int) * B, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        b->counts_fresh = true;
    }
    int n_max = 8, nc_max = 1;
    for (int i = 0; i < B; ++i) {
        const int ns_i = b->h_ns[i], nc_i = b->h_nc[i];
        if (!(ns_i >= 1 && ns_i <= b->ns_cap && nc_i >= 0 && nc_i <= NC_MAX)) continue;      // the kernel reports it
        if (ns_i + nc_i > n_max) n_max = ns_i + nc_i;
        if (nc_i > nc_max) nc_max = nc_i;
    }
    *n_max_out = n_max; *nc_max_out = nc_max;
    return 0;
}

// Runs the setup kernel on the staged device inputs and fetches the per-instance headers and counts.
static int run_setup(bqb_batch *b, int check_max, cudaStream_t s) {
    const int B = b->n_inst;
    SetupArgs a;
    a.ns = b->d_ns; a.nc = b->d_nc; a.x_s = b->d_xs; a.l_s = b->d_ls; a.x_c = b->d_xc; a.hyp = b->d_hyp; a.prior = b->d_prior;
    a.in_stride = b->ns_cap; a.check_max = check_max; a.models = b->d_models; a.lay = b->lay;
    a.work = b->d_work; a.work_stride = b->work_stride;
    int n_max, nc_max;
    const int rc = staged_sizes(b, s, &n_max, &nc_max);
    if (rc) return rc;
    a.n_max = n_max; a.nc_max = nc_max;
    a.kind = b->kind; a.period = b->d_period; a.xo = b->d_xo; a.pxo = b->d_pxo; a.n_xo = b->n_xo; a.xo_stride = b->xo_stride;
    a.wp = b->d_wp; a.gz = b->d_gz;
    a.alpha = b->d_alpha; a.alpha_stride = b->alpha_stride;
    a.inst_list = nullptr;
    // Launch groups: the setup kernel runs two CTAs per SM while two instances fit its shared memory, sized for the
    // LARGEST instance of a launch.  When a few large instances (many surviving candidates) would push a big batch into the
    // one-CTA variant, they get a launch of their own (C5: the last rounds, profiles/c5_rounds_r02.txt).
    std::vector<int> order;
    int n_small_grp = B;
    if (B > 4 * b->sm_count) {
        const int lim = setup2_two_cta_limit(nc_max);
        if (lim > 0 && n_max > lim) {
            std::vector<int> big;
            order.reserve(B);
            for (int i = 0; i < B; ++i) {
                const int n_i = b->h_ns[i] + b->h_nc[i];
                (n_i <= lim ? order : big).push_back(i);
            }
            n_small_grp = (int)order.size();
            if (n_small_grp >= B - B / 4 && !big.empty()) {            // worth it: at least 3/4 of the batch stays small
                order.insert(order.end(), big.begin(), big.end());
                if (!b->d_inst_list) CU(cudaMalloc(&b->d_inst_list, sizeof(int) * B));
                CU(cudaMemcpyAsync(b->d_inst_list, order.data(), sizeof(int) * B, cudaMemcpyHostToDevice, s));
                CU(cudaStreamSynchronize(s));                          // `order` is a local
                a.inst_list = b->d_inst_list;
            } else {
                n_small_grp = B;
            }
            if (a.inst_list) {
                int nm = 8;
                for (int k = 0; k < n_small_grp; ++k) { const int i = order[k]; nm = std::max(nm, b->h_ns[i] + b->h_nc[i]); }
                a.n_max = nm;                                          // of the first group; the second uses the batch maximum
            }
        }
    }
    for (int g0 = 0, g1 = n_small_grp; g0 < B; g0 = g1, g1 = B) {      // one or two groups
        if (g0 > 0) a.n_max = n_max;
        for (int i0 = g0; i0 < g1; i0 += b->work_inst) {
            const int cnt = (g1 - i0 < b->work_inst) ? g1 - i0 : b->work_inst;
            a.inst0 = i0;
            CU(launch_setup2(a, cnt, s));
            b->launches++;
        }
    }
    // headers (Z_mean, Z_var, log_lh, status) and l_c rows back to the host: gathered on the device, one contiguous copy
    constexpr int IW = H_COUNT + NC_MAX;
    CU(launch_pack_info(b->d_models, b->lay.total, b->lay.off_lc, B, b->d_info, s));
    b->launches++;
    CU(cudaMemcpyAsync(b->h_info, b->d_info, sizeof(double) * (size_t)B * IW, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    for (int i = 0; i < B; ++i) {
        memcpy(&b->h_hdr[(size_t)i * H_COUNT], b->h_info + (size_t)i * IW, sizeof(double) * H_COUNT);
        memcpy(&b->h_lc[(size_t)i * NC_MAX], b->h_info + (size_t)i * IW + H_COUNT, sizeof(double) * NC_MAX);
    }
    b->ndb_max = 1; b->nb_max = 1; b->nrow_max = 2;
    for (int i = 0; i < B; ++i) {
        const int d = (b->h_nc[i] + 2 + 7) / 8, nbk = (b->h_ns[i] + 7) / 8, nr = b->h_nc[i] + 2;
        if (d > b->ndb_max) b->ndb_max = d;
        if (nbk > b->nb_max) b->nb_max = nbk;
        if (nr > b->nrow_max) b->nrow_max = nr;
    }
    b->ready = true;
    return 0;
}

int bqb_batch_stage(bqb_batch *b, const int *ns, const double *x_s, const double *l_s, int in_stride, const double *hyp,
                    const double *prior, void *stream) {
    if (!b || !ns || !x_s || !l_s || !hyp || !prior) return fail(BQB_EINVAL, "bqb_batch_stage: null argument");
    if (in_stride < 1 || in_stride > b->ns_cap) return fail(BQB_EINVAL, "bqb_batch_stage: in_stride exceeds the batch capacity");
    for (int i = 0; i < b->n_inst; ++i)
        if (ns[i] < 1 || ns[i] > in_stride) return fail(BQB_EINVAL, "bqb_batch_stage: ns out of range");
    cudaStream_t s = (cudaStream_t)stream;
    CU(cudaSetDevice(b->device));
    const int B = b->n_inst;
    CU(cudaMemcpyAsync(b->d_ns, ns, sizeof(int) * B, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpy2DAsync(b->d_xs, sizeof(double) * b->ns_cap, x_s, sizeof(double) * in_stride, sizeof(double) * in_stride, B,
                         cudaMemcpyHostToDevice, s));
    CU(cudaMemcpy2DAsync(b->d_ls, sizeof(double) * b->ns_cap, l_s, sizeof(double) * in_stride, sizeof(double) * in_stride, B,
                         cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(b->d_hyp, hyp, sizeof(double) * (size_t)B * 6, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(b->d_prior, prior, sizeof(double) * (size_t)B * 3, cudaMemcpyHostToDevice, s));
    CU(cudaStreamSynchronize(s));          // the host arrays may be pageable and are free to change after this call
    b->staged = true;
    b->ready = false;
    b->counts_fresh = false;
    return 0;
}

int bqb_batch_setup(bqb_batch *b, const int *ns, const int *nc, const double *x_s, const double *l_s, int in_stride,
                    const double *x_c, const double *hyp, const double *prior, int check_max, void *stream) {
    if (!b || !nc) return fail(BQB_EINVAL, "bqb_batch_setup: null argument");
    int rc = bqb_batch_stage(b, ns, x_s, l_s, in_stride, hyp, prior, stream);
    if (rc) return rc;
    for (int i = 0; i < b->n_inst; ++i) {
        if (nc[i] < 0 || nc[i] > NC_MAX) return fail(BQB_EUNSUPPORTED, "bqb_batch_setup: more than 16 candidates");
        if (nc[i] > 0 && !x_c) return fail(BQB_EINVAL, "bqb_batch_setup: x_c is null");
    }
    cudaStream_t s = (cudaStream_t)stream;
    const int B = b->n_inst;
    CU(cudaMemcpyAsync(b->d_nc, nc, sizeof(int) * B, cudaMemcpyHostToDevice, s));
    if (x_c) CU(cudaMemcpyAsync(b->d_xc, x_c, sizeof(double) * (size_t)B * NC_MAX, cudaMemcpyHostToDevice, s));
    for (int i = 0; i < B; ++i) { b->h_ns[i] = ns[i]; b->h_nc[i] = nc[i]; }
    b->counts_fresh = true;
    return run_setup(b, check_max, s);
}

int bqb_batch_set_hypers(bqb_batch *b, const double *hyp, void *stream) {
    if (!b || !hyp) return fail(BQB_EINVAL, "bqb_batch_set_hypers: null argument");
    if (!b->staged) return fail(BQB_ESTATE, "bqb_batch_set_hypers: nothing staged (bqb_batch_stage / bqb_batch_setup first)");
    CU(cudaSetDevice(b->device));
    cudaStream_t s = (cudaStream_t)stream;
    CU(cudaMemcpyAsync(b->d_hyp, hyp, sizeof(double) * (size_t)b->n_inst * 6, cudaMemcpyHostToDevice, s));
    CU(cudaStreamSynchronize(s));          // the host array may be pageable and is free to change after this call
    b->ready = false;
    return 0;
}

// The gradient kernel on rows of (instance, hyper-parameters [, periods]): kind 0 writes grad [n][6], kind 1 grad [n][8]
static int run_llgrad(bqb_batch *b, int kind, const char *who, const double *hyp, const double *period, const int *inst,
                      int n_eval, int check_max, double *log_lh_out, double *grad_out, int *status_out, void *stream) {
    const std::string name(who);
    if (!b) return fail(BQB_EINVAL, name + ": null batch");
    if (!b->staged) return fail(BQB_ESTATE, name + ": nothing staged (bqb_batch_stage / bqb_batch_setup first)");
    if (n_eval < 0 || (n_eval > 0 && (!hyp || (kind && !period) || !log_lh_out || !grad_out || !status_out)) ||
        (!inst && n_eval > b->n_inst))
        return fail(BQB_EINVAL, name + ": bad arguments");
    for (int e = 0; inst && e < n_eval; ++e)
        if (inst[e] < 0 || inst[e] >= b->n_inst) return fail(BQB_EINVAL, name + ": instance index out of range");
    if (b->kind != kind)
        return fail(BQB_EUNSUPPORTED, name + (kind ? ": the batch does not use the periodic kernel (bqb_batch_set_approx)"
                                                   : ": only the Gaussian kernel is supported"));
    if (n_eval == 0) return 0;
    CU(cudaSetDevice(b->device));
    cudaStream_t s = (cudaStream_t)stream;
    LLGradArgs a;
    int rc = staged_sizes(b, s, &a.n_max, &a.nc_max);
    if (rc) return rc;
    if ((size_t)n_eval > b->cap_llg) {
        for (void *p : {(void *)b->d_llg_hyp, (void *)b->d_llg_out, (void *)b->d_llg_inst, (void *)b->d_llg_period}) if (p) cudaFree(p);
        b->d_llg_hyp = b->d_llg_out = b->d_llg_period = nullptr; b->d_llg_inst = nullptr; b->cap_llg = 0;
        CU(cudaMalloc(&b->d_llg_hyp, sizeof(double) * 6 * (size_t)n_eval));
        CU(cudaMalloc(&b->d_llg_out, sizeof(double) * LLG_OUT_PERIODIC * (size_t)n_eval));
        CU(cudaMalloc(&b->d_llg_period, sizeof(double) * 2 * (size_t)n_eval));
        CU(cudaMalloc(&b->d_llg_inst, sizeof(int) * (size_t)n_eval));
        b->cap_llg = n_eval;
    }
    CU(cudaMemcpyAsync(b->d_llg_hyp, hyp, sizeof(double) * 6 * (size_t)n_eval, cudaMemcpyHostToDevice, s));
    if (kind) CU(cudaMemcpyAsync(b->d_llg_period, period, sizeof(double) * 2 * (size_t)n_eval, cudaMemcpyHostToDevice, s));
    if (inst) CU(cudaMemcpyAsync(b->d_llg_inst, inst, sizeof(int) * (size_t)n_eval, cudaMemcpyHostToDevice, s));
    a.ns = b->d_ns; a.nc = b->d_nc; a.x_s = b->d_xs; a.l_s = b->d_ls; a.x_c = b->d_xc; a.in_stride = b->ns_cap;
    a.hyp = b->d_llg_hyp; a.inst = inst ? b->d_llg_inst : nullptr; a.e0 = 0; a.check_max = check_max;
    a.work = b->d_work; a.work_stride = b->work_stride; a.out = b->d_llg_out;
    a.period = kind ? b->d_llg_period : nullptr;
    int launches = 0;
    const cudaError_t e = launch_llgrad(a, n_eval, b->work_inst, s, &launches, kind);
    b->launches += launches;
    CU(e);
    const int nout = kind ? LLG_OUT_PERIODIC : LLG_OUT, ngrad = nout - 2;
    std::vector<double> h((size_t)n_eval * nout);
    CU(cudaMemcpyAsync(h.data(), b->d_llg_out, sizeof(double) * h.size(), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    for (int r = 0; r < n_eval; ++r) {
        const double *o = &h[(size_t)r * nout];
        log_lh_out[r] = o[0];
        memcpy(grad_out + (size_t)r * ngrad, o + 1, sizeof(double) * ngrad);
        status_out[r] = (int)o[nout - 1];
    }
    return 0;
}

int bqb_batch_log_lh_grad(bqb_batch *b, const double *hyp, const int *inst, int n_eval, int check_max, double *log_lh_out,
                          double *grad_out, int *status_out, void *stream) {
    return run_llgrad(b, 0, "bqb_batch_log_lh_grad", hyp, nullptr, inst, n_eval, check_max, log_lh_out, grad_out, status_out,
                      stream);
}

int bqb_batch_log_lh_grad_periodic(bqb_batch *b, const double *hyp, const double *period, const int *inst, int n_eval,
                                   int check_max, double *log_lh_out, double *grad_out, int *status_out, void *stream) {
    return run_llgrad(b, 1, "bqb_batch_log_lh_grad_periodic", hyp, period, inst, n_eval, check_max, log_lh_out, grad_out,
                      status_out, stream);
}

int bqb_batch_set_periods(bqb_batch *b, const double *period, void *stream) {
    if (!b || !period) return fail(BQB_EINVAL, "bqb_batch_set_periods: null argument");
    if (b->kind != 1 || !b->d_period)
        return fail(BQB_ESTATE, "bqb_batch_set_periods: the batch does not use the periodic kernel (bqb_batch_set_approx first)");
    CU(cudaSetDevice(b->device));
    cudaStream_t s = (cudaStream_t)stream;
    CU(cudaMemcpyAsync(b->d_period, period, sizeof(double) * (size_t)b->n_inst * 2, cudaMemcpyHostToDevice, s));
    CU(cudaStreamSynchronize(s));          // the host array may be pageable and is free to change after this call
    b->ready = false;
    return 0;
}

int bqb_batch_set_approx(bqb_batch *b, int kernel_kind, const double *period, const double *xo, const double *p_xo, int n_xo,
                         long long xo_stride, int force_generic) {
    if (!b || kernel_kind < 0 || kernel_kind > 1 || n_xo < 0 || (n_xo == 1) || xo_stride < 0)
        return fail(BQB_EINVAL, "bqb_batch_set_approx: bad arguments");
    if (kernel_kind == 1 && !period) return fail(BQB_EINVAL, "bqb_batch_set_approx: the periodic kernel needs its periods");
    if (n_xo > 0 && (!xo || !p_xo || (xo_stride != 0 && xo_stride < n_xo))) return fail(BQB_EINVAL, "bqb_batch_set_approx: bad grid");
    CU(cudaSetDevice(b->device));
    const size_t B = (size_t)b->n_inst;
    for (double **p : {&b->d_period, &b->d_xo, &b->d_pxo, &b->d_wp, &b->d_gz}) { if (*p) cudaFree(*p); *p = nullptr; }
    if (kernel_kind == 1) {
        CU(cudaMalloc(&b->d_period, sizeof(double) * B * 2));
        CU(cudaMemcpy(b->d_period, period, sizeof(double) * B * 2, cudaMemcpyHostToDevice));
    }
    if (n_xo > 0) {
        const size_t n_grid = xo_stride ? B * (size_t)xo_stride : (size_t)n_xo;
        CU(cudaMalloc(&b->d_xo, sizeof(double) * n_grid));
        CU(cudaMalloc(&b->d_pxo, sizeof(double) * n_grid));
        CU(cudaMemcpy(b->d_xo, xo, sizeof(double) * n_grid, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(b->d_pxo, p_xo, sizeof(double) * n_grid, cudaMemcpyHostToDevice));
        CU(cudaMalloc(&b->d_wp, sizeof(double) * B * (size_t)n_xo));
        CU(cudaMalloc(&b->d_gz, sizeof(double) * (size_t)b->work_inst * (size_t)n_xo));
    }
    b->kind = kernel_kind; b->n_xo = n_xo; b->xo_stride = xo_stride;
    b->generic = kernel_kind != 0 || n_xo > 0 || force_generic != 0 || b->big_class;
    b->ready = false;
    return 0;
}

int bqb_batch_setup_device(bqb_batch *b, int check_max, void *stream) {
    if (!b || !b->staged) return fail(BQB_ESTATE, "bqb_batch_setup_device: nothing staged (bqb_batch_stage / bqb_batch_setup first)");
    CU(cudaSetDevice(b->device));
    return run_setup(b, check_max, (cudaStream_t)stream);
}

int bqb_batch_seed_candidates(bqb_batch *b, const unsigned *seeds, void *stream) {
    if (!b || !seeds) return fail(BQB_EINVAL, "bqb_batch_seed_candidates: null argument");
    CU(cudaSetDevice(b->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int B = b->n_inst;
    if (!b->d_mt) CU(cudaMalloc(&b->d_mt, sizeof(unsigned) * 624 * (size_t)B));
    if (!b->d_mti) CU(cudaMalloc(&b->d_mti, sizeof(int) * B));
    unsigned *d_seeds = nullptr;
    CU(cudaMalloc(&d_seeds, sizeof(unsigned) * B));
    CU(cudaMemcpyAsync(d_seeds, seeds, sizeof(unsigned) * B, cudaMemcpyHostToDevice, s));
    cudaError_t e = launch_mt_seed(d_seeds, b->d_mt, b->d_mti, B, s);
    b->launches++;
    cudaStreamSynchronize(s);
    cudaFree(d_seeds);
    CU(e);
    return 0;
}

int bqb_batch_rng_get(bqb_batch *b, unsigned *mt_out, int *pos_out) {
    if (!b || !b->d_mt || !mt_out || !pos_out) return fail(BQB_ESTATE, "bqb_batch_rng_get: generators were not seeded");
    CU(cudaSetDevice(b->device));
    CU(cudaMemcpy(mt_out, b->d_mt, sizeof(unsigned) * 624 * (size_t)b->n_inst, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(pos_out, b->d_mti, sizeof(int) * b->n_inst, cudaMemcpyDeviceToHost));
    return 0;
}

int bqb_batch_rng_set(bqb_batch *b, const unsigned *mt, const int *pos) {
    if (!b || !mt || !pos) return fail(BQB_EINVAL, "bqb_batch_rng_set: null argument");
    CU(cudaSetDevice(b->device));
    if (!b->d_mt) CU(cudaMalloc(&b->d_mt, sizeof(unsigned) * 624 * (size_t)b->n_inst));
    if (!b->d_mti) CU(cudaMalloc(&b->d_mti, sizeof(int) * b->n_inst));
    CU(cudaMemcpy(b->d_mt, mt, sizeof(unsigned) * 624 * (size_t)b->n_inst, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(b->d_mti, pos, sizeof(int) * b->n_inst, cudaMemcpyHostToDevice));
    return 0;
}

int bqb_batch_draw_candidates(bqb_batch *b, int n_candidate, void *stream) {
    if (!b || !b->staged) return fail(BQB_ESTATE, "bqb_batch_draw_candidates: nothing staged");
    if (!b->d_mt) return fail(BQB_ESTATE, "bqb_batch_draw_candidates: generators were not seeded");
    if (n_candidate < 0 || n_candidate > NC_MAX) return fail(BQB_EUNSUPPORTED, "bqb_batch_draw_candidates: more than 16 candidates");
    CU(cudaSetDevice(b->device));
    CU(launch_draw_candidates(b->d_xs, b->d_ns, b->ns_cap, b->d_hyp, b->d_prior, b->d_mt, b->d_mti, n_candidate, b->d_xc,
                              b->d_nc, b->n_inst, (cudaStream_t)stream));
    b->launches++;
    b->ready = false;
    b->counts_fresh = false;
    return 0;
}

int bqb_batch_draw_candidates_wrapped(bqb_batch *b, int n_candidate, void *stream) {
    if (!b || !b->staged) return fail(BQB_ESTATE, "bqb_batch_draw_candidates_wrapped: nothing staged");
    if (!b->d_mt) return fail(BQB_ESTATE, "bqb_batch_draw_candidates_wrapped: generators were not seeded");
    if (b->kind != 1 || !b->d_period)
        return fail(BQB_ESTATE, "bqb_batch_draw_candidates_wrapped: the batch does not use the periodic kernel (bqb_batch_set_approx first)");
    if (n_candidate < 0 || n_candidate > NC_MAX)
        return fail(BQB_EUNSUPPORTED, "bqb_batch_draw_candidates_wrapped: more than 16 candidates");
    CU(cudaSetDevice(b->device));
    CU(launch_draw_candidates_wrapped(b->d_xs, b->d_ns, b->ns_cap, b->d_period, b->d_prior, b->d_mt, b->d_mti, n_candidate,
                                      b->d_xc, b->d_nc, b->n_inst, (cudaStream_t)stream));
    b->launches++;
    b->ready = false;
    b->counts_fresh = false;
    return 0;
}

int bqb_batch_add_observations(bqb_batch *b, const double *d_x_new, const double *d_l_new, void *stream) {
    if (!b || !b->staged) return fail(BQB_ESTATE, "bqb_batch_add_observations: nothing staged");
    if (!d_x_new || !d_l_new) return fail(BQB_EINVAL, "bqb_batch_add_observations: null argument");
    CU(cudaSetDevice(b->device));
    cudaStream_t s = (cudaStream_t)stream;
    if (!b->d_overflow) CU(cudaMalloc(&b->d_overflow, sizeof(int)));
    CU(cudaMemsetAsync(b->d_overflow, 0, sizeof(int), s));
    CU(launch_add_observations(b->d_xs, b->d_ls, b->d_ns, b->ns_cap, b->d_prior, d_x_new, d_l_new, b->n_inst, b->d_overflow, s));
    b->launches++;
    b->ready = false;
    b->counts_fresh = false;
    int ov = 0;
    CU(cudaMemcpyAsync(&ov, b->d_overflow, sizeof(int), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    if (ov) return fail(BQB_EUNSUPPORTED, "bqb_batch_add_observations: an instance is at the batch's observation capacity");
    return 0;
}

int bqb_batch_get_staged(bqb_batch *b, int *ns, int *nc, double *x_s, double *l_s, double *x_c) {
    if (!b || !b->staged) return fail(BQB_ESTATE, "bqb_batch_get_staged: nothing staged");
    CU(cudaSetDevice(b->device));
    const size_t B = b->n_inst;
    if (ns) CU(cudaMemcpy(ns, b->d_ns, sizeof(int) * B, cudaMemcpyDeviceToHost));
    if (nc) CU(cudaMemcpy(nc, b->d_nc, sizeof(int) * B, cudaMemcpyDeviceToHost));
    if (x_s) CU(cudaMemcpy(x_s, b->d_xs, sizeof(double) * B * b->ns_cap, cudaMemcpyDeviceToHost));
    if (l_s) CU(cudaMemcpy(l_s, b->d_ls, sizeof(double) * B * b->ns_cap, cudaMemcpyDeviceToHost));
    if (x_c) CU(cudaMemcpy(x_c, b->d_xc, sizeof(double) * B * NC_MAX, cudaMemcpyDeviceToHost));
    return 0;
}

int bqb_batch_capacity(bqb_batch *b) { return b ? b->ns_cap : BQB_EINVAL; }

int bqb_batch_info(bqb_batch *b, double *Z_mean, double *Z_var, double *log_lh, int *status, double *l_c) {
    if (!b || !b->ready) return fail(BQB_ESTATE, "bqb_batch_info: batch was not set up");
    for (int i = 0; i < b->n_inst; ++i) {
        const double *h = &b->h_hdr[(size_t)i * H_COUNT];
        if (Z_mean) Z_mean[i] = h[H_ZM];
        if (Z_var) Z_var[i] = h[H_ZV];
        if (log_lh) log_lh[i] = h[H_LOGLH];
        if (status) status[i] = (int)h[H_STATUS];
    }
    if (l_c) memcpy(l_c, b->h_lc.data(), sizeof(double) * b->h_lc.size());
    return 0;
}

// the tensor-core kernels (Gaussian kernel, closed-form integrals) or the generic kernel (bqb_batch_set_approx).
// `first`: the instance at which a.models begins.  The single-instance entry points pass that instance's own model block
// with inst0 = 0, so the generic kernel's per-instance grid and trapezoid weights must begin at the same instance.
static cudaError_t score_dispatch(bqb_batch *b, ScoreArgs &a, int n_inst, cudaStream_t s, int *grid_x = nullptr, int first = 0) {
    if (b->generic) {
        a.xo = b->d_xo ? b->d_xo + (size_t)first * b->xo_stride : nullptr;
        a.wp = b->d_wp ? b->d_wp + (size_t)first * b->n_xo : nullptr;
        a.n_xo = b->n_xo; a.xo_stride = b->xo_stride;
        return launch_score_generic(a, n_inst, s, grid_x);
    }
    return launch_score(a, n_inst, b->sm_count, s, grid_x);
}

// The scoring arguments that come from the batch, with a.models beginning at instance `first`
static ScoreArgs score_args(const bqb_batch *b, int first = 0) {
    ScoreArgs a;
    a.models = b->d_models + (size_t)first * b->lay.total; a.lay = b->lay; a.exp_tab = b->d_tab;
    a.cut_arg = b->cut_arg; a.work = b->d_work_ctr;
    a.nb_max = b->nb_max; a.nrow_max = b->nrow_max; a.ndb_max = b->ndb_max;
    return a;
}

// Instances [first, first + count) of a batch-wide launch (a.models at instance 0), in launches of at most 32768
// instances: gridDim.y is limited to 65535
static int score_chunks(bqb_batch *b, ScoreArgs &a, int first, int count, cudaStream_t s) {
    for (int i0 = first; i0 < first + count; i0 += 32768) {
        a.inst0 = i0;
        CU(score_dispatch(b, a, std::min(first + count - i0, 32768), s));
        b->launches++;
    }
    return 0;
}

static int check_ready(bqb_batch *b, const char *who) {
    if (!b || !b->ready) return fail(BQB_ESTATE, std::string(who) + ": batch was not set up");
    for (int i = 0; i < b->n_inst; ++i)
        if ((int)b->h_hdr[(size_t)i * H_COUNT + H_STATUS] != SETUP_OK)
            return fail(BQB_ENUMERIC, std::string(who) + ": an instance failed setup (see bqb_batch_info status)");
    return 0;
}

static int score_device_impl(bqb_batch *b, const double *d_x_a, long long xa_stride, int na, double *d_esm, double *d_em,
                             int *d_status, long long out_stride, int *d_flags, const int *d_perm, void *stream, int first = 0,
                             int count = -1, int xa_group = 1);

int bqb_score_device(bqb_batch *b, const double *d_x_a, long long xa_stride, int na, double *d_esm, double *d_em,
                     int *d_status, long long out_stride, int *d_flags, void *stream) {
    return score_device_impl(b, d_x_a, xa_stride, na, d_esm, d_em, d_status, out_stride, d_flags, nullptr, stream);
}

int bqb_score_device_range(bqb_batch *b, int inst0, int n_inst, const double *d_x_a, long long xa_stride, int na, double *d_esm,
                           double *d_em, int *d_status, long long out_stride, int *d_flags, void *stream) {
    if (!b || inst0 < 0 || n_inst < 1 || inst0 + n_inst > b->n_inst) return fail(BQB_EINVAL, "bqb_score_device_range: bad instance range");
    return score_device_impl(b, d_x_a, xa_stride, na, d_esm, d_em, d_status, out_stride, d_flags, nullptr, stream, inst0, n_inst);
}

int bqb_score_device_grouped(bqb_batch *b, int inst0, int n_inst, const double *d_x_a, long long xa_stride, int xa_group, int na,
                             double *d_esm, double *d_em, int *d_status, long long out_stride, int *d_flags, void *stream) {
    if (!b || inst0 < 0 || n_inst < 1 || inst0 + n_inst > b->n_inst) return fail(BQB_EINVAL, "bqb_score_device_grouped: bad instance range");
    if (xa_group < 1 || inst0 % xa_group) return fail(BQB_EINVAL, "bqb_score_device_grouped: inst0 must be a multiple of xa_group >= 1");
    return score_device_impl(b, d_x_a, xa_stride, na, d_esm, d_em, d_status, out_stride, d_flags, nullptr, stream, inst0, n_inst,
                             xa_group);
}

// A query vector "looks sorted" if ~2000 evenly spaced samples are ascending at stride 1 and at the sampling stride.
// Only performance depends on the answer (sorted or not, every point is scored and lands in its own slot).
static bool looks_sorted(const double *x, int n) {
    const int stride = n / 2048 > 1 ? n / 2048 : 1;
    for (int i = 0; i + stride < n; i += stride)
        if (!(x[i] <= x[i + 1]) || !(x[i] <= x[i + stride])) return false;
    return true;
}

// Sorts the n points at d_x on stream s: b->d_xsorted ascending, b->d_perm their original positions.
static int sort_query(bqb_batch *b, const double *d_x, int n, cudaStream_t s) {
    if ((size_t)n > b->cap_sort) {
        if (b->d_xsorted) cudaFree(b->d_xsorted);
        if (b->d_perm) cudaFree(b->d_perm);
        if (b->d_iota) cudaFree(b->d_iota);
        b->d_xsorted = nullptr; b->d_perm = b->d_iota = nullptr; b->cap_sort = 0;
        CU(cudaMalloc(&b->d_xsorted, sizeof(double) * n));
        CU(cudaMalloc(&b->d_perm, sizeof(int) * n));
        CU(cudaMalloc(&b->d_iota, sizeof(int) * n));
        b->cap_sort = n;
    }
    size_t need = 0;
    CU(sort_points(d_x, n, b->d_xsorted, b->d_iota, b->d_perm, nullptr, &need, s));
    if (need > b->cap_sort_tmp) {
        if (b->d_sort_tmp) cudaFree(b->d_sort_tmp);
        b->d_sort_tmp = nullptr; b->cap_sort_tmp = 0;
        CU(cudaMalloc(&b->d_sort_tmp, need));
        b->cap_sort_tmp = need;
    }
    need = b->cap_sort_tmp;
    CU(sort_points(d_x, n, b->d_xsorted, b->d_iota, b->d_perm, b->d_sort_tmp, &need, s));
    b->launches += 2;
    return 0;
}
constexpr int PRESORT_MIN = 8192;     // below this the penalty of unsorted points is not worth a sort
// automatic mode: only for the classes where unsorted points cost more than the sort and the lost copy/compute overlap
// (measured through BQ.expected_Z_var, 10^6 shuffled points: ns = 256 6.8 -> 2.1 ms with the sort, ns = 64 0.84 -> 1.11 ms)
static bool want_presort(const bqb_batch *b, const double *x, int n) {
    if (n < PRESORT_MIN || b->presort == 0) return false;
    if (b->presort == 2) return true;
    return b->ns_cap >= 128 && !looks_sorted(x, n);
}

// Instances [first, first + count) (count < 0: all).  The per-instance rows of x_a / esm / em / status / flags are relative
// to `first` (row 0 belongs to instance `first`), so a caller can walk a large batch through one chunk-sized buffer.
static int score_device_impl(bqb_batch *b, const double *d_x_a, long long xa_stride, int na, double *d_esm, double *d_em,
                             int *d_status, long long out_stride, int *d_flags, const int *d_perm, void *stream, int first, int count,
                             int xa_group) {
    int rc = check_ready(b, "bqb_score_device");
    if (rc) return rc;
    if (!d_x_a || !d_esm || na < 0 || out_stride < na) return fail(BQB_EINVAL, "bqb_score_device: bad arguments");
    if (na == 0) return 0;
    if (count < 0) count = b->n_inst - first;
    CU(cudaSetDevice(b->device));
    ScoreArgs a = score_args(b);
    a.x_a = d_x_a - (size_t)(first / xa_group) * xa_stride; a.xa_stride = xa_stride; a.xa_group = xa_group; a.na = na;
    a.esm = d_esm - (size_t)first * out_stride; a.em = d_em ? d_em - (size_t)first * out_stride : nullptr;
    a.status = d_status ? d_status - (size_t)first * out_stride : nullptr; a.out_stride = out_stride;
    a.flags = d_flags ? d_flags - first : nullptr; a.perm = d_perm;
    if (d_flags) CU(cudaMemsetAsync(d_flags, 0, sizeof(int) * count, (cudaStream_t)stream));
    return score_chunks(b, a, first, count, (cudaStream_t)stream);
}

int bqb_predict_device(bqb_batch *b, const double *d_x, long long x_stride, int na, double *d_l_mean, double *d_v_log_l,
                       long long out_stride, void *stream) {
    int rc = check_ready(b, "bqb_predict_device");
    if (rc) return rc;
    if (b->generic) return fail(BQB_EUNSUPPORTED, "bqb_predict_device: not offered with bqb_batch_set_approx (generic kernel)");
    if (!d_x || !d_l_mean || !d_v_log_l || na < 0 || out_stride < na) return fail(BQB_EINVAL, "bqb_predict_device: bad arguments");
    if (na == 0) return 0;
    CU(cudaSetDevice(b->device));
    ScoreArgs a = score_args(b);
    a.x_a = d_x; a.xa_stride = x_stride; a.na = na;
    a.esm = d_l_mean; a.em = d_v_log_l; a.out_stride = out_stride; a.predict = 1;
    return score_chunks(b, a, 0, b->n_inst, (cudaStream_t)stream);
}

static int grow(bqb_batch *b, size_t n_xa, size_t n_out) {
    if (n_xa > b->cap_xa) {
        if (b->d_xa) cudaFree(b->d_xa);
        CU(cudaMalloc(&b->d_xa, sizeof(double) * n_xa));
        b->cap_xa = n_xa;
    }
    if (n_out > b->cap_out) {
        if (b->d_esm) cudaFree(b->d_esm);
        if (b->d_em) cudaFree(b->d_em);
        if (b->d_st) cudaFree(b->d_st);
        CU(cudaMalloc(&b->d_esm, sizeof(double) * n_out));
        CU(cudaMalloc(&b->d_em, sizeof(double) * n_out));
        CU(cudaMalloc(&b->d_st, sizeof(int) * n_out));
        b->cap_out = n_out;
    }
    return 0;
}

int bqb_score_host(bqb_batch *b, const double *x_a, long long xa_stride, int na, double *esm, double *em, int *status) {
    int rc = check_ready(b, "bqb_score_host");
    if (rc) return rc;
    if (!x_a || !esm || na < 0) return fail(BQB_EINVAL, "bqb_score_host: bad arguments");
    if (na == 0) return 0;
    CU(cudaSetDevice(b->device));
    const size_t B = b->n_inst;
    const size_t n_xa = xa_stride ? B * (size_t)xa_stride : (size_t)na;
    rc = grow(b, n_xa, B * (size_t)na);
    if (rc) return rc;
    cudaStream_t s = 0;
    CU(cudaMemcpyAsync(b->d_xa, x_a, sizeof(double) * n_xa, cudaMemcpyHostToDevice, s));
    const double *d_x = b->d_xa;
    const int *d_perm = nullptr;
    if (xa_stride == 0 && want_presort(b, x_a, na)) {
        rc = sort_query(b, b->d_xa, na, s);          // points in arbitrary order defeat band skipping: score them sorted
        if (rc) return rc;
        d_x = b->d_xsorted; d_perm = b->d_perm;
    }
    rc = score_device_impl(b, d_x, xa_stride, na, b->d_esm, em ? b->d_em : nullptr, status ? b->d_st : nullptr, na, nullptr,
                           d_perm, s);
    if (rc) return rc;
    CU(cudaMemcpyAsync(esm, b->d_esm, sizeof(double) * B * na, cudaMemcpyDeviceToHost, s));
    if (em) CU(cudaMemcpyAsync(em, b->d_em, sizeof(double) * B * na, cudaMemcpyDeviceToHost, s));
    if (status) CU(cudaMemcpyAsync(status, b->d_st, sizeof(int) * B * na, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    return 0;
}

// Page-locked host memory (cudaHostAlloc / cudaHostRegister, e.g. a pinned torch tensor) is mapped into the device
// address space under unified addressing: the scoring kernel can read its query points from it and write its
// results to it directly, so the transfer overlaps the arithmetic point by point instead of chunk by chunk.
static bool mapped_host(const void *p, void **dev) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    if (at.type != cudaMemoryTypeHost || !at.devicePointer) return false;
    *dev = at.devicePointer;
    return true;
}

int bqb_predict_host(bqb_batch *b, const double *x, long long x_stride, int na, double *l_mean, double *v_log_l) {
    int rc = check_ready(b, "bqb_predict_host");
    if (rc) return rc;
    if (!x || !l_mean || !v_log_l || na < 0) return fail(BQB_EINVAL, "bqb_predict_host: bad arguments");
    if (na == 0) return 0;
    CU(cudaSetDevice(b->device));
    const size_t B = b->n_inst;
    const size_t n_x = x_stride ? B * (size_t)x_stride : (size_t)na;
    rc = grow(b, n_x, B * (size_t)na);
    if (rc) return rc;
    cudaStream_t s = 0;
    CU(cudaMemcpyAsync(b->d_xa, x, sizeof(double) * n_x, cudaMemcpyHostToDevice, s));
    rc = bqb_predict_device(b, b->d_xa, x_stride, na, b->d_esm, b->d_em, na, s);
    if (rc) return rc;
    CU(cudaMemcpyAsync(l_mean, b->d_esm, sizeof(double) * B * na, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(v_log_l, b->d_em, sizeof(double) * B * na, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    return 0;
}

// The checks of bqb_predict_rows_device / _host.  *listed: rows listed (rows null: every instance), 0 when there is nothing to
// do (na = 0 or an empty list: the pointers are not looked at, as in bqb_expected_var_rows_device)
static int predict_rows_check(bqb_batch *b, const char *who, const int *rows, int n_rows, const void *x, long long x_stride, int na,
                              const void *l_mean, const void *v_log_l, long long out_stride, int *listed) {
    const std::string name(who);
    if (!b) return fail(BQB_EINVAL, name + ": null batch");
    if (na < 0 || out_stride < na || x_stride < 0 || (x_stride && x_stride < na) || (rows && n_rows < 0))
        return fail(BQB_EINVAL, name + ": bad arguments");
    for (int i = 0; rows && i < n_rows; ++i)
        if (rows[i] < 0 || rows[i] >= b->n_inst) return fail(BQB_EINVAL, name + ": row out of range");
    *listed = (na == 0) ? 0 : rows ? n_rows : b->n_inst;
    if (*listed == 0) return 0;
    int rc = check_ready(b, who);
    if (rc) return rc;
    if (!x || !l_mean || !v_log_l) return fail(BQB_EINVAL, name + ": bad arguments");
    return 0;
}

static int predict_rows_launch(bqb_batch *b, const int *rows, int listed, const double *d_x, long long x_stride, int na,
                               double *d_l_mean, double *d_v_log_l, long long out_stride, cudaStream_t s) {
    CU(cudaSetDevice(b->device));
    PredictArgs a;
    a.models = b->d_models; a.lay = b->lay; a.alpha = b->d_alpha; a.alpha_stride = b->alpha_stride;
    a.x = d_x; a.x_stride = x_stride; a.na = na;
    a.l_mean = d_l_mean; a.v_log_l = d_v_log_l; a.out_stride = out_stride;
    if (rows) {
        if ((size_t)listed > b->cap_rows) {
            if (b->d_rows) cudaFree(b->d_rows);
            b->d_rows = nullptr; b->cap_rows = 0;
            CU(cudaMalloc(&b->d_rows, sizeof(int) * (size_t)listed));
            b->cap_rows = listed;
        }
        // (pageable `rows` are staged before the copy call returns; page-locked ones are read when the stream gets there)
        CU(cudaMemcpyAsync(b->d_rows, rows, sizeof(int) * (size_t)listed, cudaMemcpyHostToDevice, s));
        a.rows = b->d_rows;
    }
    for (int r0 = 0; r0 < listed; r0 += 32768) {               // gridDim.y is limited to 65535
        a.row0 = r0;
        CU(launch_predict(a, std::min(listed - r0, 32768), s));
        b->launches++;
    }
    return 0;
}

int bqb_predict_rows_device(bqb_batch *b, const int *rows, int n_rows, const double *d_x, long long x_stride, int na,
                            double *d_l_mean, double *d_v_log_l, long long out_stride, void *stream) {
    int listed = 0;
    int rc = predict_rows_check(b, "bqb_predict_rows_device", rows, n_rows, d_x, x_stride, na, d_l_mean, d_v_log_l, out_stride,
                                &listed);
    if (rc || listed == 0) return rc;
    return predict_rows_launch(b, rows, listed, d_x, x_stride, na, d_l_mean, d_v_log_l, out_stride, (cudaStream_t)stream);
}

int bqb_predict_rows_host(bqb_batch *b, const int *rows, int n_rows, const double *x, long long x_stride, int na, double *l_mean,
                          double *v_log_l) {
    int listed = 0;
    int rc = predict_rows_check(b, "bqb_predict_rows_host", rows, n_rows, x, x_stride, na, l_mean, v_log_l, na, &listed);
    if (rc || listed == 0) return rc;
    CU(cudaSetDevice(b->device));
    const size_t B = b->n_inst;
    const size_t n_x = x_stride ? B * (size_t)x_stride : (size_t)na;
    rc = grow(b, n_x, B * (size_t)na);
    if (rc) return rc;
    cudaStream_t s = 0;
    CU(cudaMemcpyAsync(b->d_xa, x, sizeof(double) * n_x, cudaMemcpyHostToDevice, s));
    rc = predict_rows_launch(b, rows, listed, b->d_xa, x_stride, na, b->d_esm, b->d_em, na, s);
    if (rc) return rc;
    if (!rows) {
        CU(cudaMemcpyAsync(l_mean, b->d_esm, sizeof(double) * B * na, cudaMemcpyDeviceToHost, s));
        CU(cudaMemcpyAsync(v_log_l, b->d_em, sizeof(double) * B * na, cudaMemcpyDeviceToHost, s));
    }
    for (int i = 0; rows && i < listed; ++i) {                   // only the listed rows of the outputs are written
        const size_t o = (size_t)rows[i] * na;
        CU(cudaMemcpyAsync(l_mean + o, b->d_esm + o, sizeof(double) * na, cudaMemcpyDeviceToHost, s));
        CU(cudaMemcpyAsync(v_log_l + o, b->d_em + o, sizeof(double) * na, cudaMemcpyDeviceToHost, s));
    }
    CU(cudaStreamSynchronize(s));
    return 0;
}

int bqb_alpha_read(bqb_batch *b, int inst, double *out) {
    if (!b || !b->ready || inst < 0 || inst >= b->n_inst || !out) return fail(BQB_EINVAL, "bqb_alpha_read: bad arguments");
    const double *h = &b->h_hdr[(size_t)inst * H_COUNT];
    if ((int)h[H_STATUS] != SETUP_OK) return fail(BQB_ENUMERIC, "bqb_alpha_read: the instance failed setup");
    CU(cudaSetDevice(b->device));
    const int n = (int)h[H_NS] + (int)h[H_NC];
    CU(cudaMemcpy(out, b->d_alpha + (size_t)inst * b->alpha_stride, sizeof(double) * n, cudaMemcpyDeviceToHost));
    return 0;
}

int bqb_expected_var_host(bqb_batch *b, int inst, const double *x_a, int na, double *out, int *flags_out) {
    int rc = check_ready(b, "bqb_expected_var_host");
    if (rc) return rc;
    if (inst < 0 || inst >= b->n_inst || !x_a || !out || na < 0) return fail(BQB_EINVAL, "bqb_expected_var_host: bad arguments");
    if (na == 0) { if (flags_out) *flags_out = 0; return 0; }
    CU(cudaSetDevice(b->device));
    static const int zero_copy_env = getenv("BQB_ZERO_COPY") ? atoi(getenv("BQB_ZERO_COPY")) : 1;
    const int zero_copy = zero_copy_env && b->zero_copy;
    const bool presort = want_presort(b, x_a, na);
    void *dx = nullptr, *dout = nullptr;
    const bool in_mapped = !presort && zero_copy && mapped_host(x_a, &dx);      // a vector to be sorted is staged on the device
    const bool out_mapped = !presort && zero_copy && mapped_host(out, &dout);
    if (!in_mapped || !out_mapped) {
        rc = grow(b, (size_t)na, (size_t)b->n_inst * na);
        if (rc) return rc;
    }
    if (!b->d_flags) CU(cudaMalloc(&b->d_flags, sizeof(int) * b->n_inst));
    if (!b->h_flags) CU(cudaMallocHost(&b->h_flags, sizeof(int)));
    for (cudaStream_t &st : b->pipe) if (!st) CU(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    // Buffers that are not page-locked go through device staging in chunks that alternate between two streams, so
    // that the H2D copy of one chunk, the kernels of another and the D2H copy of a third overlap.
    static const int min_chunk = getenv("BQB_PIPE_CHUNK") ? atoi(getenv("BQB_PIPE_CHUNK")) : (1 << 18);
    int nchunk = ((in_mapped && out_mapped) || presort) ? 1 : na / min_chunk;
    if (nchunk < 1) nchunk = 1;
    if (nchunk > 8) nchunk = 8;
    int per = ((na + nchunk - 1) / nchunk + 255) & ~255;
    const bool zc = in_mapped && out_mapped;              // one launch; status words come back through mapped memory too
    if (zc && !b->h_cta_flags) CU(cudaMallocHost(&b->h_cta_flags, sizeof(int) * 4096));
    if (!zc) CU(cudaMemsetAsync(b->d_flags, 0, sizeof(int) * b->n_inst, b->pipe[0]));
    if (nchunk > 1) CU(cudaStreamSynchronize(b->pipe[0]));
    int zc_grid = 0;
    ScoreArgs a = score_args(b, inst);
    a.flags = zc ? nullptr : b->d_flags; a.cta_flags = zc ? b->h_cta_flags : nullptr;
    int c = 0;
    for (int lo = 0; lo < na; lo += per, ++c) {
        const int n = (na - lo < per) ? na - lo : per;
        cudaStream_t s = b->pipe[c & 1];
        if (in_mapped) {
            a.x_a = (const double *)dx + lo;
        } else {
            CU(cudaMemcpyAsync(b->d_xa + lo, x_a + lo, sizeof(double) * n, cudaMemcpyHostToDevice, s));
            a.x_a = b->d_xa + lo;
            if (presort) {                               // single chunk: sort, score ascending, results back through perm
                rc = sort_query(b, b->d_xa, na, s);
                if (rc) return rc;
                a.x_a = b->d_xsorted; a.perm = b->d_perm;
            }
        }
        a.na = n; a.out_stride = n;
        if (out_mapped) {
            // fused epilogue: Zm^2 + Zv - esm written straight into the caller's page-locked array
            a.esm = nullptr; a.ev = (double *)dout + lo;
            a.part_val = b->d_red_val + 2048 * (c & 1); a.part_idx = b->d_red_idx + 2048 * (c & 1);
            CU(score_dispatch(b, a, 1, s, &zc_grid, inst));
            b->launches += 1;
        } else {
            a.esm = b->d_esm + lo; a.ev = nullptr;
            CU(score_dispatch(b, a, 1, s, nullptr, inst));
            CU(launch_expected_var_rows(b->d_models, b->lay.total, inst, 1, b->d_esm + lo, n, n, b->d_em + lo, n, s));
            b->launches += 2;
            CU(cudaMemcpyAsync(out + lo, b->d_em + lo, sizeof(double) * n, cudaMemcpyDeviceToHost, s));
        }
    }
    if (nchunk > 1) CU(cudaStreamSynchronize(b->pipe[1]));
    if (zc) {
        CU(cudaStreamSynchronize(b->pipe[0]));
        int fl = 0;
        for (int i = 0; i < zc_grid && i < 4096; ++i) fl |= b->h_cta_flags[i];
        if (flags_out) *flags_out = fl;
        return 0;
    }
    CU(cudaMemcpyAsync(b->h_flags, b->d_flags, sizeof(int), cudaMemcpyDeviceToHost, b->pipe[0]));
    CU(cudaStreamSynchronize(b->pipe[0]));
    if (flags_out) *flags_out = *b->h_flags;
    return 0;
}

int bqb_mean_neg_device(bqb_batch *b, const double *d_esm, long long stride, long long na, double *d_loss, void *stream) {
    if (!b || !d_esm || !d_loss || na < 0) return fail(BQB_EINVAL, "bqb_mean_neg_device: bad arguments");
    CU(cudaSetDevice(b->device));
    CU(launch_sum_neg_groups(d_esm, stride, 1, b->n_inst, na, d_loss, 0, true, (cudaStream_t)stream));
    b->launches++;
    return 0;
}

int bqb_sum_neg_accum_device(bqb_batch *b, const double *d_esm, long long stride, int n_rows, long long na, double *d_acc, void *stream) {
    if (!b || !d_esm || !d_acc || na < 0 || n_rows < 0 || stride < na) return fail(BQB_EINVAL, "bqb_sum_neg_accum_device: bad arguments");
    if (na == 0 || n_rows == 0) return 0;
    CU(cudaSetDevice(b->device));
    CU(launch_sum_neg_groups(d_esm, stride, 1, n_rows, na, d_acc, 0, false, (cudaStream_t)stream));
    b->launches++;
    return 0;
}

int bqb_sum_neg_accum_groups_device(bqb_batch *b, const double *d_esm, long long stride, int n_groups, int group_size, long long na,
                                    double *d_acc, long long acc_stride, void *stream) {
    if (!b || na < 0 || n_groups < 0 || group_size < 0) return fail(BQB_EINVAL, "bqb_sum_neg_accum_groups_device: bad arguments");
    if (na == 0 || n_groups == 0 || group_size == 0) return 0;                  // nothing is read or written
    if (!d_esm || !d_acc || stride < na || (n_groups > 1 && acc_stride < na))
        return fail(BQB_EINVAL, "bqb_sum_neg_accum_groups_device: bad arguments");
    CU(cudaSetDevice(b->device));
    CU(launch_sum_neg_groups(d_esm, stride, n_groups, group_size, na, d_acc, acc_stride, false, (cudaStream_t)stream));
    b->launches++;
    return 0;
}

int bqb_expected_var_device(bqb_batch *b, int inst, const double *d_esm, long long na, double *d_out, void *stream) {
    int rc = check_ready(b, "bqb_expected_var_device");
    if (rc) return rc;
    if (inst < 0 || inst >= b->n_inst || !d_esm || !d_out) return fail(BQB_EINVAL, "bqb_expected_var_device: bad arguments");
    CU(cudaSetDevice(b->device));
    CU(launch_expected_var_rows(b->d_models, b->lay.total, inst, 1, d_esm, na, na, d_out, na, (cudaStream_t)stream));
    b->launches++;
    return 0;
}

int bqb_expected_var_rows_device(bqb_batch *b, int inst0, int n_inst, const double *d_esm, long long esm_stride, long long na,
                                 double *d_out, long long out_stride, void *stream) {
    if (!b || inst0 < 0 || n_inst < 0 || inst0 > b->n_inst - n_inst)
        return fail(BQB_EINVAL, "bqb_expected_var_rows_device: bad instance range");
    if (na < 0 || esm_stride < na || out_stride < na) return fail(BQB_EINVAL, "bqb_expected_var_rows_device: bad arguments");
    if (na == 0 || n_inst == 0) return 0;
    int rc = check_ready(b, "bqb_expected_var_rows_device");
    if (rc) return rc;
    if (!d_esm || !d_out) return fail(BQB_EINVAL, "bqb_expected_var_rows_device: bad arguments");
    CU(cudaSetDevice(b->device));
    CU(launch_expected_var_rows(b->d_models, b->lay.total, inst0, n_inst, d_esm, esm_stride, na, d_out, out_stride,
                                (cudaStream_t)stream));
    b->launches++;
    return 0;
}

int bqb_argmin_device(bqb_batch *b, const double *d_v, long long n, double *min_out, long long *idx_out, void *stream) {
    if (!b || !d_v || n < 1 || !min_out || !idx_out) return fail(BQB_EINVAL, "bqb_argmin_device: bad arguments");
    CU(cudaSetDevice(b->device));
    cudaStream_t s = (cudaStream_t)stream;
    CU(launch_argmin(d_v, n, b->d_red_val, b->d_red_idx, b->sm_count, 0, nullptr, s));
    b->launches += 2;
    CU(cudaMemcpyAsync(min_out, b->d_red_val, sizeof(double), cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(idx_out, b->d_red_idx, sizeof(long long), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    return 0;
}

int bqb_argmin_pair_device(bqb_batch *b, const double *d_v, long long n, long long offset, double *d_pair, void *stream) {
    if (!b || !d_v || n < 1 || !d_pair) return fail(BQB_EINVAL, "bqb_argmin_pair_device: bad arguments");
    CU(cudaSetDevice(b->device));
    CU(launch_argmin(d_v, n, b->d_red_val, b->d_red_idx, b->sm_count, offset, d_pair, (cudaStream_t)stream));
    b->launches += 2;
    return 0;
}

// The scoring launch of a choose_next step: esm and the fused expected variance of instance `inst`, with the per-CTA
// (min, first index) partials of the expected variance in b->d_red_val / b->d_red_idx and their number in *grid_x
static int choose_step_score(bqb_batch *b, int inst, const double *d_x_a, int na, double *d_esm, double *d_ev, cudaStream_t s,
                             int *grid_x) {
    CU(cudaSetDevice(b->device));
    ScoreArgs a = score_args(b, inst);
    a.x_a = d_x_a; a.na = na; a.esm = d_esm; a.out_stride = na;
    a.ev = d_ev; a.part_val = b->d_red_val; a.part_idx = b->d_red_idx;
    CU(score_dispatch(b, a, 1, s, grid_x, inst));
    return 0;
}

int bqb_choose_step_device(bqb_batch *b, int inst, const double *d_x_a, int na, double *d_esm, double *d_ev, long long offset,
                           double *d_pair, void *stream) {
    int rc = check_ready(b, "bqb_choose_step_device");
    if (rc) return rc;
    if (inst < 0 || inst >= b->n_inst || !d_x_a || !d_esm || !d_ev || !d_pair || na < 1)
        return fail(BQB_EINVAL, "bqb_choose_step_device: bad arguments");
    cudaStream_t s = (cudaStream_t)stream;
    int grid_x = 0;
    rc = choose_step_score(b, inst, d_x_a, na, d_esm, d_ev, s, &grid_x);
    if (rc) return rc;
    CU(launch_argmin_partials(b->d_red_val, b->d_red_idx, grid_x, offset, d_pair, s));
    b->launches += 2;
    return 0;
}

int bqb_choose_step_exchange(bqb_batch *b, int inst, const double *d_x_a, int na, double *d_esm, double *d_ev, long long offset,
                             long long cyclic_block, void *const *peer_slots, int world, int rank, unsigned long long seq,
                             double *out4, void *stream) {
    int rc = check_ready(b, "bqb_choose_step_exchange");
    if (rc) return rc;
    if (inst < 0 || inst >= b->n_inst || !d_x_a || !d_ev || !peer_slots || !out4 || na < 1 || world < 1 || world > 16 || rank < 0 ||
        rank >= world || seq == 0 || cyclic_block < 0)
        return fail(BQB_EINVAL, "bqb_choose_step_exchange: bad arguments");
    cudaStream_t s = (cudaStream_t)stream;
    int grid_x = 0;
    rc = choose_step_score(b, inst, d_x_a, na, d_esm, d_ev, s, &grid_x);
    if (rc) return rc;
    CU(launch_argmin_exchange(b->d_red_val, b->d_red_idx, grid_x, offset, cyclic_block, peer_slots, world, rank, seq, out4, s));
    b->launches += 2;
    return 0;
}

int bqb_argmin_rows_device(bqb_batch *b, const double *d_v, long long stride, long long n, double *d_min,
                           long long *d_idx, void *stream) {
    if (!b || !d_v || n < 1 || stride < n || !d_min || !d_idx) return fail(BQB_EINVAL, "bqb_argmin_rows_device: bad arguments");
    CU(cudaSetDevice(b->device));
    CU(launch_argmin_rows(d_v, stride, n, b->n_inst, d_min, d_idx, (cudaStream_t)stream));
    b->launches++;
    return 0;
}

int bqb_argmin_ties_rows_device(bqb_batch *b, const double *d_v, long long stride, long long n, const double *d_min,
                                const double *d_u, long long *d_idx, long long *d_count, void *stream) {
    if (!b || !d_v || n < 1 || stride < n || !d_min || !d_u || !d_idx)
        return fail(BQB_EINVAL, "bqb_argmin_ties_rows_device: bad arguments");
    CU(cudaSetDevice(b->device));
    CU(launch_argmin_ties_rows(d_v, stride, n, b->n_inst, d_min, d_u, d_idx, d_count, (cudaStream_t)stream));
    b->launches++;
    return 0;
}

unsigned long long bqb_launch_count(bqb_batch *b) { return b ? b->launches : 0; }

int bqb_batch_set_presort(bqb_batch *b, int mode) {
    if (!b || mode < 0 || mode > 2) return fail(BQB_EINVAL, "bqb_batch_set_presort: mode must be 0 (never), 1 (automatic) or 2 (always)");
    b->presort = mode;
    return 0;
}

int bqb_batch_set_zero_copy(bqb_batch *b, int enable) {
    if (!b) return fail(BQB_EINVAL, "bqb_batch_set_zero_copy: null batch");
    b->zero_copy = enable ? 1 : 0;
    return 0;
}

int bqb_batch_set_cutoff(bqb_batch *b, double cut_arg) {
    if (!b || !(cut_arg > 0)) return fail(BQB_EINVAL, "bqb_batch_set_cutoff: cut_arg must be positive (INFINITY = dense)");
    b->cut_arg = cut_arg;
    return 0;
}

int bqb_batch_work_counter(bqb_batch *b, int enable, unsigned long long *dmma_out) {
    if (!b) return fail(BQB_EINVAL, "bqb_batch_work_counter: null batch");
    CU(cudaSetDevice(b->device));
    if (dmma_out) {
        *dmma_out = 0;
        if (b->d_work_ctr) CU(cudaMemcpy(dmma_out, b->d_work_ctr, sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    }
    if (enable && !b->d_work_ctr) CU(cudaMalloc(&b->d_work_ctr, sizeof(unsigned long long)));
    if (b->d_work_ctr) CU(cudaMemset(b->d_work_ctr, 0, sizeof(unsigned long long)));
    if (!enable && b->d_work_ctr) { cudaFree(b->d_work_ctr); b->d_work_ctr = nullptr; }
    return 0;
}

int bqb_model_doubles(bqb_batch *b) { return b ? b->lay.total : 0; }

int bqb_model_read(bqb_batch *b, int inst, double *out) {
    if (!b || !b->ready || inst < 0 || inst >= b->n_inst || !out) return fail(BQB_EINVAL, "bqb_model_read: bad arguments");
    CU(cudaSetDevice(b->device));
    CU(cudaMemcpy(out, b->d_models + (size_t)inst * b->lay.total, sizeof(double) * b->lay.total, cudaMemcpyDeviceToHost));
    return 0;
}

}  // extern "C"
