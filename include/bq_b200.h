/* bq_b200.h — C-ABI of the B200-native expected-variance active-sampling path of
 * jhamrick/bayesian-quadrature (v0.2.0).
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch / numpy / C++ types.  It
 * replaces the native entry points the reference's Python layer binds for this path
 * (Cython typed-memoryview functions, SURVEY.md §8(b)); each function below names the reference
 * interface it stands in for (paths relative to the reference repository).
 *
 * A *batch* is B independent model instances — one BQ problem under one hyper-parameter set
 * each — resident in HBM.  The reference evaluates one query point per call of
 * BQ._esm_and_em (bayesian_quadrature/bq.py:447-527); here ONE call scores a whole vector of
 * query points for every instance of the batch.
 *
 * All floating point data is IEEE float64.  Return value: 0 = success; < 0 = argument/state
 * error (BQB_E*, the reference raises ValueError via la.value_error, linalg_c.pyx:49-50);
 * > 0 = a cudaError_t.  bqb_last_error() gives the message (thread local).  Functions never
 * throw and never retain caller pointers.
 */
#ifndef BQ_B200_H
#define BQ_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define BQB_EINVAL (-1)        /* bad argument (reference: ValueError) */
#define BQB_EUNSUPPORTED (-2)  /* outside device limits: ns > 512, nc > 16, not sm_100 */
#define BQB_ESTATE (-3)        /* batch not set up */
#define BQB_ENUMERIC (-4)      /* an instance failed setup (reference: numpy.linalg.LinAlgError) */

/* per-point status bits written by the scoring kernel; the host shim turns them into the
 * reference's exceptions / warnings */
#define BQB_ST_OK 0
#define BQB_ST_SHORTCUT 1   /* bq.py:456-459: x_a isclose to an observation -> (Z_mean^2, Z_mean) */
#define BQB_ST_NOTPD 2      /* bq.py:481-490: bordered matrix not PD (LinAlgError) -> (Z_mean^2, Z_mean) */
#define BQB_ST_ESM_INF 4    /* bq.py:522-523: logger.warn */
#define BQB_ST_EM_INF 8     /* bq.py:524-525: logger.warn */
#define BQB_ST_ESM_BAD 16   /* bq.py:514-517: RuntimeError */
#define BQB_ST_EM_BAD 32    /* bq.py:518-520: RuntimeError */
#define BQB_ST_XA_BAD 64    /* bq.py:451-452: ValueError */

/* per-instance setup status (bqb_batch_info) */
#define BQB_SETUP_OK 0
#define BQB_SETUP_KTL_NOTPD 1       /* gp_log_l.Kxx not positive definite (LinAlgError) */
#define BQB_SETUP_KL_NOTPD 2        /* gp_l.Kxx not positive definite (LinAlgError) */
#define BQB_SETUP_MEAN_TOO_LARGE 3  /* bq.py:945-947 LinAlgError("GP mean is too large") */
#define BQB_SETUP_BAD_INPUT 4       /* non-finite x / l <= 0 / non-positive hyper-parameters (ValueError) */

#define BQB_NC_MAX 16               /* row stride of every x_c / l_c array */

typedef struct bqb_batch bqb_batch;

const char *bqb_last_error(void);
int bqb_version(void);
int bqb_device_count(int *count);

/* Padded observation capacity the library would use for `ns` observations (16, 64, 128, 160, 256, or 512: the last class
 * runs on the generic plain-FP64 scoring kernel only, see bqb_batch_set_approx), or
 * BQB_EUNSUPPORTED. */
int bqb_ns_capacity(int ns);

/* Allocates a batch of n_inst instances on CUDA device `device`, each able to hold up to ns_max
 * observations and BQB_NC_MAX candidates.  Stands in for BQ.__init__ state allocation
 * (bq.py:55-92) plus the `gp` objects of BQ.init (bq.py:147-165). */
int bqb_batch_create(bqb_batch **out, int device, int n_inst, int ns_max);
void bqb_batch_destroy(bqb_batch *b);

/* Uploads the instances (HOST pointers) and runs the setup kernel.  Per instance i:
 *   ns[i], nc[i]            observation / candidate counts
 *   x_s, l_s [i*in_stride]  observation locations and (positive) likelihood values
 *   x_c [i*BQB_NC_MAX]      candidate locations (already drawn/filtered on the host, bq.py:967-991)
 *   hyp [i*6]               h_tl, w_tl, s_tl, h_l, w_l, s_l   (GP params of bq.py:132-165)
 *   prior [i*3]             x_mean, x_var, candidate_thresh   (options of bq.py:94-127)
 * Computes on device what the reference obtains from the `gp` package and linalg_c:
 * tl_s = log l_s (bq.py:73), K_tl and its Cholesky factor (gp.Lxx; linalg_c.cho_factor
 * linalg_c.pyx:55), l_c = exp(gp_log_l.mean(x_c)) (bq.py:985, :949), the factor of K_l(x_sc, x_sc),
 * alpha_l (gp.inv_Kxx_y), Z_mean (bq_c.Z_mean bq_c.pyx:157), Z_var (bq_c.Z_var bq_c.pyx:264 with
 * gauss_c.int_int_K1_K2_K1 gauss_c.pyx:416 and gauss_c.int_K1_K2 gauss_c.pyx:235) and
 * gp_log_l.log_lh + gp_l.log_lh (bq.py:546).  check_max != 0 applies the guard of
 * BQ._set_gp_log_l_params (bq.py:942-947).  Synchronises `stream` (a cudaStream_t, may be 0). */
int bqb_batch_setup(bqb_batch *b, const int *ns, const int *nc, const double *x_s, const double *l_s,
                    int in_stride, const double *x_c, const double *hyp, const double *prior,
                    int check_max, void *stream);

/* ---- device-resident active sampling over a batch of independent problems (SURVEY.md §8(f).2) ----------------
 * The observations of every instance stay in HBM between rounds: a round is
 *   bqb_score_device -> bqb_argmin_rows_device -> (caller evaluates the likelihood at the chosen points)
 *   -> bqb_batch_add_observations -> bqb_batch_draw_candidates -> bqb_batch_setup_device.
 *
 * bqb_batch_stage: the upload half of bqb_batch_setup (HOST pointers; x_s / l_s rows of in_stride doubles are
 * stored with the batch's own row stride bqb_batch_capacity(), so observations can be appended in place). */
int bqb_batch_stage(bqb_batch *b, const int *ns, const double *x_s, const double *l_s, int in_stride,
                    const double *hyp, const double *prior, void *stream);
/* Replaces the hyper-parameters hyp [n_inst][6] (HOST pointer) of a staged batch and nothing else: the next
 * bqb_batch_setup_device refactorises the same observations and candidates under them.  This is what one evaluation of
 * the hyper-parameter log-density costs (BQ._make_llh_params, bq.py:533-552: _set_gp_log_l_params :933-957 +
 * _set_gp_l_params :959-965 + gp.log_lh) -- no buffer is reallocated, nothing but 48 bytes per instance is uploaded. */
int bqb_batch_set_hypers(bqb_batch *b, const double *hyp, void *stream);
/* Value and gradient of the joint log marginal likelihood that BQ._make_llh_params / BQ.fit_hypers maximise
 * (bq.py:533-562: gp_log_l.log_lh + gp_l.log_lh after l_c is recomputed from the candidates) for n_eval rows, each an
 * instance under its own hyper-parameters.  hyp [n_eval][6] (h, w, s of gp_log_l, then of gp_l), inst [n_eval] (instance
 * of each row; NULL: row e is instance e, n_eval <= n_inst) and the outputs are HOST arrays: log_lh_out [n_eval],
 * grad_out [n_eval][6] (d log_lh / d of the six hyper-parameters, in the order of hyp) and status_out [n_eval] (the setup
 * status codes; a row that is not OK has log_lh -inf and a NaN gradient).  check_max applies the "GP mean is too large"
 * guard (bq.py:942-947).  Reads the staged observations and candidates; leaves the model blocks and the batch's own
 * hyper-parameters untouched, so the scoring model stays valid.  Gaussian kernel only (BQB_EUNSUPPORTED after
 * bqb_batch_set_approx with the periodic kernel); BQB_ESTATE when nothing is staged.  Synchronises `stream`. */
int bqb_batch_log_lh_grad(bqb_batch *b, const double *hyp, const int *inst, int n_eval, int check_max, double *log_lh_out,
                          double *grad_out, int *status_out, void *stream);
/* bqb_batch_log_lh_grad for a batch of the periodic kernel (bqb_batch_set_approx with kernel_kind 1): each row also has
 * its periods, period [n_eval][2] (p of gp_log_l, then of gp_l; HOST array), and grad_out is [n_eval][8]: d log_lh / d
 * (h_tl, w_tl, s_tl, h_l, w_l, s_l, p_tl, p_l).  BQB_EUNSUPPORTED unless the batch uses the periodic kernel; BQB_ESTATE
 * when nothing is staged.  Synchronises `stream`. */
int bqb_batch_log_lh_grad_periodic(bqb_batch *b, const double *hyp, const double *period, const int *inst, int n_eval,
                                   int check_max, double *log_lh_out, double *grad_out, int *status_out, void *stream);
/* The periodic twin of bqb_batch_set_hypers: replaces the periods period [n_inst][2] (HOST pointer) of a batch of the
 * periodic kernel and nothing else (the grids of bqb_batch_set_approx stay as they are).  BQB_ESTATE when the batch does
 * not use the periodic kernel. */
int bqb_batch_set_periods(bqb_batch *b, const double *period, void *stream);
/* Non-Gaussian kernels and the trapezoid approximation.  Replaces gp.PeriodicKernel as used by bq.py:139-165 and
 * bq_c.approx_Z_mean (bq_c.pyx:216-261), approx_Z_var (:358-422), approx_expected_squared_mean_and_mean (:538-598),
 * i.e. what BQ does when options['use_approx'] is set (bq.py:251-252, :310-311, :498-510).
 *   kernel_kind 0: gp.GaussianKernel(h, w);  1: gp.PeriodicKernel(h, w, p) with period[i] = {p of gp_log_l, p of gp_l}
 *   n_xo > 0: the integrals over the prior are trapezoid sums over the grid xo with prior density p_xo (HOST arrays,
 *             [n_xo] shared by all instances when xo_stride = 0, else [n_inst][xo_stride]); n_xo = 0: closed forms
 *             (Gaussian kernel only).
 *   force_generic != 0 runs the plain-FP64 scoring kernel even for the Gaussian / closed-form case (cross-checks).
 * Takes effect at the next setup call; afterwards every scoring entry point except bqb_predict_device / _host works as
 * before (bqb_predict_rows_* predicts for every batch). */
int bqb_batch_set_approx(bqb_batch *b, int kernel_kind, const double *period, const double *xo, const double *p_xo, int n_xo,
                         long long xo_stride, int force_generic);
/* The setup half: runs the setup kernel on whatever is staged on the device (after bqb_batch_stage /
 * bqb_batch_add_observations / bqb_batch_draw_candidates).  Stands in for BQ.init (bq.py:132-171) of every
 * instance.  Synchronises `stream`. */
int bqb_batch_setup_device(bqb_batch *b, int check_max, void *stream);
/* One numpy.random.RandomState(seeds[i]) per instance (MT19937 seeded like numpy's legacy integer seeding),
 * resident on the device; bqb_batch_rng_get / _set copy the generator states ([624][n_inst] words, word-major, and
 * the n_inst positions) to / from HOST arrays, e.g. to continue a stream that the host started. */
int bqb_batch_seed_candidates(bqb_batch *b, const unsigned *seeds, void *stream);
int bqb_batch_rng_get(bqb_batch *b, unsigned *mt_out, int *pos_out);
int bqb_batch_rng_set(bqb_batch *b, const unsigned *mt, const int *pos);
/* BQ._choose_candidates (bq.py:967-991) for every instance on the device: n_candidate draws of
 * np.random.uniform(x_s.min() - w_tl, x_s.max() + w_tl) from the instance's generator (bit-identical to numpy),
 * bq_c.filter_candidates (bq_c.pyx:601-650) with the instance's candidate_thresh, np.sort of the survivors. */
int bqb_batch_draw_candidates(bqb_batch *b, int n_candidate, void *stream);
/* bqb_batch_draw_candidates with the periodic kernel's wrapped range (bq.py:217-218): the draws are
 * np.random.uniform(-pi p_tl, pi p_tl) with p_tl the instance's period of gp_log_l; the filter and sort are the same.
 * BQB_ESTATE when the batch does not use the periodic kernel. */
int bqb_batch_draw_candidates_wrapped(bqb_batch *b, int n_candidate, void *stream);
/* BQ.add_observation (bq.py:683-701) for every instance: DEVICE arrays d_x_new / d_l_new [n_inst]; the new point
 * is averaged into the nearest observation when closer than candidate_thresh, appended otherwise.  Returns
 * BQB_EUNSUPPORTED if an instance is already at bqb_batch_capacity() observations.  Synchronises `stream`. */
int bqb_batch_add_observations(bqb_batch *b, const double *d_x_new, const double *d_l_new, void *stream);
/* Copies the staged state to HOST arrays (any may be NULL): ns, nc [n_inst]; x_s, l_s [n_inst][capacity];
 * x_c [n_inst][BQB_NC_MAX]. */
int bqb_batch_get_staged(bqb_batch *b, int *ns, int *nc, double *x_s, double *l_s, double *x_c);
int bqb_batch_capacity(bqb_batch *b);

/* Per-instance results of the setup (HOST output arrays of n_inst entries, any may be NULL;
 * l_c is [n_inst][BQB_NC_MAX]).  Z_mean / Z_var replace BQ._exact_Z_mean (bq.py:268-291) and
 * BQ._exact_Z_var (bq.py:329-348). */
int bqb_batch_info(bqb_batch *b, double *Z_mean, double *Z_var, double *log_lh, int *status, double *l_c);

/* Scores na query points for every instance; replaces the loop of
 * BQ.expected_squared_mean_and_mean (bq.py:425-445) over BQ._esm_and_em (bq.py:447-527) and
 * bq_c.expected_squared_mean_and_mean (bq_c.pyx:493-535).
 *   x_a        query points: shared by all instances (xa_stride = 0) or one row per instance
 *   esm, em    outputs [n_inst][out_stride] (em may be NULL): expected squared mean / expected mean
 *   status     per-point BQB_ST_* bits [n_inst][out_stride] (may be NULL)
 *   d_flags    [n_inst] OR of all status bits of an instance (may be NULL): lets the caller skip
 *              the status vector unless something other than BQB_ST_OK happened
 * _device: DEVICE pointers, asynchronous on `stream`.  _host: HOST pointers (out_stride = na);
 * copies in, scores, copies out and synchronises. */
int bqb_score_device(bqb_batch *b, const double *d_x_a, long long xa_stride, int na, double *d_esm,
                     double *d_em, int *d_status, long long out_stride, int *d_flags, void *stream);
int bqb_score_host(bqb_batch *b, const double *x_a, long long xa_stride, int na, double *esm, double *em,
                   int *status);

/* bqb_score_device for the instances [inst0, inst0 + n_inst) only.  Row 0 of x_a (when xa_stride != 0), esm, em, status and
 * d_flags belongs to instance inst0: a batch of many hyper-parameter sets (bq.py:640-652) can be walked through one
 * chunk-sized score buffer. */
int bqb_score_device_range(bqb_batch *b, int inst0, int n_inst, const double *d_x_a, long long xa_stride, int na, double *d_esm,
                           double *d_em, int *d_status, long long out_stride, int *d_flags, void *stream);

/* bqb_score_device_range where xa_group consecutive instances share one query row: instance i reads row
 * (i - inst0) / xa_group of x_a (when xa_stride != 0).  The S hyper-parameter samples of a problem (bq.py:640-652) are scored
 * against that problem's grid without replicating it S times.  inst0 must be a multiple of xa_group (BQB_EINVAL otherwise),
 * so that a chunk starts on a problem boundary; esm / em / status / d_flags keep one row per instance.  Never sorts x_a. */
int bqb_score_device_grouped(bqb_batch *b, int inst0, int n_inst, const double *d_x_a, long long xa_stride, int xa_group, int na,
                             double *d_esm, double *d_em, int *d_status, long long out_stride, int *d_flags, void *stream);

/* Batched prediction at na points for every instance (SURVEY.md §8(f).4): l_mean = gp_l.mean(x), the mean of the final
 * approximation (BQ.l_mean, bq.py:177-200), and v_log_l = diag gp_log_l.cov(x), from which BQ.l_var (bq.py:202-231) is
 * max(v_log_l * l_mean^2, 0).  Same layout conventions as bqb_score_*; requires s_l = 0 (the scoring factors are those
 * of the noise-free bordered matrix, SURVEY appendix A.2) and a tensor-core batch (BQB_EUNSUPPORTED after
 * bqb_batch_set_approx or in the 512 class); bqb_predict_rows_* below has neither limit. */
int bqb_predict_device(bqb_batch *b, const double *d_x, long long x_stride, int na, double *d_l_mean,
                       double *d_v_log_l, long long out_stride, void *stream);
int bqb_predict_host(bqb_batch *b, const double *x, long long x_stride, int na, double *l_mean, double *v_log_l);

/* Prediction for any batch -- tensor-core or generic, Gaussian or periodic kernel, every capacity class, any s_l -- on the
 * instances listed in `rows`: l_mean = gp_l.mean(x) (BQ.l_mean, bq.py:177-200) and v_log_l = diag gp_log_l.cov(x), from which
 * BQ.l_var (bq.py:202-231) is max(v_log_l * l_mean^2, 0).  The mean is K_l(x, x_sc) alpha_l with the alpha_l = (K_l + s_l^2 I)^-1
 * l_sc that the setup keeps (gp_l.inv_Kxx_y, bqb_alpha_read); the variance is K_tl(x, x) - |L_tl^-1 k_tl(x)|^2.  No shortcut,
 * no jitter pattern: a non-finite point gives NaN in both outputs.
 *   rows: HOST array of n_rows instance indices (any order, repeats allowed), or null for every instance (n_rows ignored).
 *         It is copied to a batch-owned device buffer on `stream` (a page-locked array is read when the stream reaches
 *         the copy), so calls on one batch must not overlap on different streams.
 *   Row i of the outputs (at i * out_stride), and row i of x when x_stride != 0, belong to INSTANCE i; rows of instances
 *   that are not listed are not written.  A point's result does not depend on the other rows or points of the call.
 * BQB_EINVAL for a null batch or pointer, n_rows < 0, a row out of range, x_stride in (0, na) or out_stride < na;
 * BQB_ESTATE / BQB_ENUMERIC when the batch is not set up / an instance failed setup.  na = 0 or an empty list does nothing
 * (the pointers and the batch's state are then not looked at).
 * The _device form takes DEVICE pointers and is asynchronous on `stream`; the _host form takes host arrays, outputs
 * [n_inst][na], and returns when they are written. */
int bqb_predict_rows_device(bqb_batch *b, const int *rows, int n_rows, const double *d_x, long long x_stride, int na,
                            double *d_l_mean, double *d_v_log_l, long long out_stride, void *stream);
int bqb_predict_rows_host(bqb_batch *b, const int *rows, int n_rows, const double *x, long long x_stride, int na,
                          double *l_mean, double *v_log_l);

/* The ns + nc entries of alpha_l = (K_l + s_l^2 I)^-1 l_sc of instance `inst` from the last setup, in model order: entry k
 * belongs to the k-th observation in ascending order for k < ns, then to candidate k - ns.  BQB_EINVAL for bad arguments or
 * a batch that is not set up, BQB_ENUMERIC when the instance failed setup. */
int bqb_alpha_read(bqb_batch *b, int inst, double *out);

/* out[p] = Z_mean^2 + Z_var - esm[p] for instance `inst` (BQ.expected_Z_var, bq.py:374-377).
 * DEVICE pointers. */
int bqb_expected_var_device(bqb_batch *b, int inst, const double *d_esm, long long na, double *d_out,
                            void *stream);

/* out[r][p] = Z_mean^2 + Z_var - esm[r][p] for the instances [inst0, inst0 + n_inst), row r of esm (at r * esm_stride) and of
 * out (at r * out_stride) belonging to instance inst0 + r: BQ.expected_Z_var of many problems (bq.py:374-377).  Z_mean and
 * Z_var are read from the model blocks on the device; every row has the bits of bqb_expected_var_host for its instance.
 * esm and out may be the same buffer.  BQB_EINVAL for a bad range or strides < na, BQB_ESTATE when the batch was not set
 * up; na = 0 or n_inst = 0 does nothing.  DEVICE pointers, asynchronous on `stream`. */
int bqb_expected_var_rows_device(bqb_batch *b, int inst0, int n_inst, const double *d_esm, long long esm_stride, long long na,
                                 double *d_out, long long out_stride, void *stream);

/* BQ.expected_Z_var(x_a) (bq.py:354-377) end to end for instance `inst`: HOST x_a in, HOST
 * out[p] = Z_mean^2 + Z_var - esm[p]; *flags_out = OR of the points' status bits.  Synchronous. */
int bqb_expected_var_host(bqb_batch *b, int inst, const double *x_a, int na, double *out, int *flags_out);

/* loss[p] = mean over instances, in instance order, of -esm[i][p]: the marginal loss of
 * BQ.choose_next (bq.py:660-662: values[0].mean(axis=0)).  DEVICE pointers. */
int bqb_mean_neg_device(bqb_batch *b, const double *d_esm, long long stride, long long na, double *d_loss,
                        void *stream);

/* d_acc[p] += -esm[0][p] - esm[1][p] - ... over n_rows rows, in row order, starting from d_acc[p]: the running form of
 * bqb_mean_neg_device.  Zero d_acc, feed the samples chunk by chunk in sample order, divide by the number of samples: the
 * same additions in the same order as values[0].mean(axis=0) (bq.py:662), without the [n_samples, na] matrix in memory; and
 * the partial sum a rank contributes when the samples are sharded across GPUs (all-reduce, then divide). */
int bqb_sum_neg_accum_device(bqb_batch *b, const double *d_esm, long long stride, int n_rows, long long na, double *d_acc,
                             void *stream);

/* Segmented bqb_sum_neg_accum_device over n_groups groups of group_size consecutive rows of esm:
 * d_acc[g][p] += -esm[g*group_size][p] - esm[g*group_size+1][p] - ... in row order (row g of d_acc at g * acc_stride).  Each
 * group performs the additions of bqb_sum_neg_accum_device, so that dividing by the number of samples gives every problem's
 * values[0].mean(axis=0) of bq.py:640-663 when the rows of a group are its hyper-parameter samples.  DEVICE pointers. */
int bqb_sum_neg_accum_groups_device(bqb_batch *b, const double *d_esm, long long stride, int n_groups, int group_size, long long na,
                                    double *d_acc, long long acc_stride, void *stream);

/* Deterministic minimum of a DEVICE vector and the FIRST index attaining it (np.min / np.argmin of
 * bq.py:663).  Results are written to HOST scalars; synchronises `stream`. */
int bqb_argmin_device(bqb_batch *b, const double *d_v, long long n, double *min_out, long long *idx_out,
                      void *stream);

/* Same reduction, left on the device for the cross-rank exchange of sharded runs: d_pair[0] = min,
 * d_pair[1] = (double)(first index + offset) (exact below 2^53).  Asynchronous on `stream`; the ranks
 * all-gather their pairs (NCCL has no MINLOC) and reduce them locally. */
int bqb_argmin_pair_device(bqb_batch *b, const double *d_v, long long n, long long offset, double *d_pair,
                           void *stream);

/* One fused step of expected-variance active sampling for instance `inst` over a (shard of a) query vector:
 * d_esm[p] (bq.py:379-402), d_ev[p] = Z_mean^2 + Z_var - esm[p] (bq.py:374-377) and the deterministic
 * (min of ev, first index + offset) pair (bq.py:663) in d_pair, in two launches (the scoring kernel carries
 * the reduction in its epilogue).  DEVICE pointers, asynchronous on `stream`. */
int bqb_choose_step_device(bqb_batch *b, int inst, const double *d_x_a, int na, double *d_esm, double *d_ev,
                           long long offset, double *d_pair, void *stream);

/* bqb_choose_step_device whose reduction also does the cross-rank exchange of sharded runs (one process per GPU): the
 * kernel that reduces this rank's partials stores its (min, first global index) pair into every rank's exchange
 * buffer -- peer_slots[r] = device pointer, valid on THIS device, of rank r's buffer of 2 * world * 4 doubles, zero
 * initialised (peer-mapped symmetric memory over NVLink; with world = 1 any device buffer) -- waits for the other
 * ranks' pairs of the same step `seq` (1, 2, 3, ... identical on all ranks) and writes out4 = {global min, global first
 * index, timed-out flag, seq}; out4 may be page-locked host memory.  The global index of local point i is i + offset
 * (contiguous shards, cyclic_block = 0) or ((i / cyclic_block) * world + rank) * cyclic_block + i % cyclic_block
 * (block-cyclic shards: every rank sees the same mix of near- and far-field points, which band skipping makes cost
 * differently).  Replaces the NCCL all-gather + local reduce + device-to-host copy of the deterministic choose_next
 * (bq.py:663) across ranks.  Asynchronous on `stream`. */
int bqb_choose_step_exchange(bqb_batch *b, int inst, const double *d_x_a, int na, double *d_esm, double *d_ev,
                             long long offset, long long cyclic_block, void *const *peer_slots, int world, int rank,
                             unsigned long long seq, double *out4, void *stream);

/* Per-instance (min, first index) of d_v [n_inst][stride] into DEVICE arrays d_min / d_idx [n_inst]: the
 * deterministic choose_next of a batch of independent problems (bq.py:663 per problem). */
int bqb_argmin_rows_device(bqb_batch *b, const double *d_v, long long stride, long long n, double *d_min,
                           long long *d_idx, void *stream);

/* The reference's random tie-break of choose_next (bq.py:664-665: np.random.choice over the points where
 * np.isclose(loss, loss.min())), per instance: with c the number of j < n where d_v[r][j] is close to d_min[r]
 * (|v - min| <= 1e-8 + 1e-5 |min| for a finite min, or v == min; NaN is close to nothing) -- d_min as
 * bqb_argmin_rows_device writes it -- d_idx[r] is the index of the k-th close point in ascending order,
 * k = min(floor(d_u[r] * c), c - 1), for a uniform d_u[r] in [0, 1).  A row without a close point (all NaN) gets
 * 0x7fffffffffffffff.  d_count [n_inst] (may be NULL) receives c.  DEVICE pointers, rows d_v [n_inst][stride];
 * asynchronous on `stream`. */
int bqb_argmin_ties_rows_device(bqb_batch *b, const double *d_v, long long stride, long long n, const double *d_min,
                                const double *d_u, long long *d_idx, long long *d_count, void *stream);

/* Band skipping (DESIGN.md): a cross-kernel element exp(-(x_a - x_s[k])^2 / 2w^2) whose exponent lies more than
 * cut_arg below the largest one of its own query point is treated as zero, and groups of four observations in which
 * every element of a 16-point sub-tile is that small are neither exponentiated nor multiplied.  Default 72
 * (e^-72 = 5e-32 of the point's leading element: below double-precision relevance for cond(K) < 1e9);
 * INFINITY (or the environment variable BQB_DENSE=1 at batch creation) runs the dense algorithm. */
int bqb_batch_set_cutoff(bqb_batch *b, double cut_arg);
/* Query vectors in arbitrary order defeat band skipping (the hull of every 32 consecutive points then spans the whole
 * domain).  The HOST entry points (bqb_score_host with a shared x_a, bqb_expected_var_host) therefore sort vectors of
 * >= 8192 points that do not look sorted (a sampled test on the host) on the device (CUB radix sort, 0.2 ms per 10^6
 * points), score them in ascending order and write every result to its original position.  mode: 0 never, 1 automatic
 * (default: batches of capacity >= 128 observations, where the sort pays), 2 always.  The DEVICE entry points never sort: pass sorted vectors for full speed. */
int bqb_batch_set_presort(bqb_batch *b, int mode);
/* bqb_expected_var_host with page-locked arrays: enable = 1 (default) lets the scoring kernel read the query points from and
 * write the results to host memory in place over PCIe (no staging copy, transfers overlap the arithmetic point by point);
 * enable = 0 stages through device buffers with chunked asynchronous copies on two streams, as for pageable arrays. */
int bqb_batch_set_zero_copy(bqb_batch *b, int enable);
/* Executed-work counter of the scoring kernel: returns in *dmma_out (may be NULL) the number of DMMA.8x8x4
 * instructions (512 flop each) executed by the launches since the last call, then clears it; enable = 1 keeps
 * counting (a few integer instructions per sub-tile), enable = 0 switches it off (the default). */
int bqb_batch_work_counter(bqb_batch *b, int enable, unsigned long long *dmma_out);

/* Introspection for tests and the bench harness. */
unsigned long long bqb_launch_count(bqb_batch *b);   /* kernels launched through this batch so far */
int bqb_model_doubles(bqb_batch *b);                  /* size of one device model block */
int bqb_model_read(bqb_batch *b, int inst, double *out);

#ifdef __cplusplus
}
#endif
#endif /* BQ_B200_H */
