// Device-resident pieces of an active-sampling round over a batch of independent problems, so that the
// observations never leave HBM between rounds (SURVEY.md §8(f).2):
//
//   add_observations_kernel   BQ.add_observation (bq.py:683-701): average the new point into the nearest observation
//                             when it is closer than candidate_thresh, append it otherwise
//   mt_seed_kernel            np.random.RandomState(seed) for a 32-bit integer seed (MT19937 init_genrand)
//   draw_candidates_kernel    BQ._choose_candidates (bq.py:967-991): n_candidate draws of
//                             np.random.uniform(x_s.min() - w_tl, x_s.max() + w_tl), bq_c.filter_candidates
//                             (bq_c.pyx:601-650), np.sort of the survivors; draw_candidates_wrapped_kernel draws
//                             on [-pi p_tl, pi p_tl] instead (the periodic kernel, bq.py:217-218)
//
// One thread per problem: each of these is a few thousand scalar operations per problem and runs once per round,
// next to a scoring launch of ~10^8 FP64 operations per problem.  The Mersenne-Twister state is stored word-major
// ([624][P]) so that the threads of a warp touch consecutive addresses.  The random stream is bit-identical to
// numpy's legacy generator: two 32-bit outputs a, b per double, (a >> 5) * 2^26 + (b >> 6) over 2^53, then
// low + (high - low) * u without FMA contraction.
#include "bq_common.cuh"

namespace bqb {

constexpr int MT_N = 624, MT_M = 397;

__global__ void mt_seed_kernel(const unsigned *__restrict__ seeds, unsigned *__restrict__ mt, int *__restrict__ mti, int P) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    unsigned s = seeds[p];
    mt[p] = s;
    for (int i = 1; i < MT_N; ++i) {
        s = 1812433253u * (s ^ (s >> 30)) + (unsigned)i;
        mt[(size_t)i * P + p] = s;
    }
    mti[p] = MT_N;
}

__device__ __forceinline__ unsigned mt_twist(unsigned u, unsigned v) {
    const unsigned y = (u & 0x80000000u) | (v & 0x7fffffffu);
    return (y >> 1) ^ ((v & 1u) ? 0x9908b0dfu : 0u);
}

__device__ unsigned mt_next(unsigned *__restrict__ mt, int &idx, int P, int p) {
    if (idx >= MT_N) {                                           // regenerate the 624 words (genrand_int32)
        int kk = 0;
        for (; kk < MT_N - MT_M; ++kk)
            mt[(size_t)kk * P + p] = mt[(size_t)(kk + MT_M) * P + p] ^ mt_twist(mt[(size_t)kk * P + p], mt[(size_t)(kk + 1) * P + p]);
        for (; kk < MT_N - 1; ++kk)
            mt[(size_t)kk * P + p] = mt[(size_t)(kk + MT_M - MT_N) * P + p] ^ mt_twist(mt[(size_t)kk * P + p], mt[(size_t)(kk + 1) * P + p]);
        mt[(size_t)(MT_N - 1) * P + p] = mt[(size_t)(MT_M - 1) * P + p] ^ mt_twist(mt[(size_t)(MT_N - 1) * P + p], mt[p]);
        idx = 0;
    }
    unsigned y = mt[(size_t)idx * P + p];
    ++idx;
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    return y;
}

// x_s, l_s: [P][stride]; ns: [P]; prior: [P][3] (candidate_thresh in slot 2).  *overflow is set when an append does
// not fit (the caller moves the batch to the next capacity class first, so this is a guard, not a path).
__global__ void add_observations_kernel(double *__restrict__ x_s, double *__restrict__ l_s, int *__restrict__ ns, int stride,
                                        const double *__restrict__ prior, const double *__restrict__ x_new,
                                        const double *__restrict__ l_new, int P, int *overflow) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    double *xs = x_s + (size_t)p * stride, *ls = l_s + (size_t)p * stride;
    const int n = ns[p];
    const double xa = x_new[p], la = l_new[p], thresh = prior[3 * p + 2];
    double dmin = INFINITY;
    int c = 0;
    for (int j = 0; j < n; ++j) {                                // np.abs(x_a - x_s).argmin(): first minimum
        const double d = fabs(xa - xs[j]);
        if (d < dmin) { dmin = d; c = j; }
    }
    if (dmin < thresh) {                                         // bq.py:685-691
        xs[c] = (xs[c] + xa) / 2.0;
        ls[c] = (ls[c] + la) / 2.0;
    } else if (n < stride) {                                     // bq.py:694-697
        xs[n] = xa;
        ls[n] = la;
        ns[p] = n + 1;
    } else {
        atomicOr(overflow, 1);
    }
}

// WRAPPED: the periodic kernel's draw on [-pi p_tl, pi p_tl] (bq.py:217-218), p_tl = period[2 p]; otherwise on
// [min x_s - w_tl, max x_s + w_tl]
template <bool WRAPPED>
__device__ __forceinline__ void draw_candidates_body(const double *__restrict__ x_s, const int *__restrict__ ns, int stride,
                                                     const double *__restrict__ hyp, const double *__restrict__ period,
                                                     const double *__restrict__ prior, unsigned *__restrict__ mt,
                                                     int *__restrict__ mti, int n_candidate, double *__restrict__ x_c,
                                                     int *__restrict__ nc, int P) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const double *xs = x_s + (size_t)p * stride;
    const int n = ns[p];
    double lo, hi, thresh;
    if (WRAPPED) {
        const double p_tl = period[2 * p];
        thresh = prior[3 * p + 2];
        lo = __dmul_rn(-M_PI, p_tl);                             // -np.pi * p, np.pi * p
        hi = __dmul_rn(M_PI, p_tl);
    } else {
        const double w_tl = hyp[6 * p + 1];
        thresh = prior[3 * p + 2];
        lo = INFINITY; hi = -INFINITY;
        for (int j = 0; j < n; ++j) { lo = fmin(lo, xs[j]); hi = fmax(hi, xs[j]); }
        lo = __dsub_rn(lo, w_tl);                                // bq.py:974-975
        hi = __dadd_rn(hi, w_tl);
    }
    const double range = __dsub_rn(hi, lo);
    double xc[NC_MAX];
    int idx = mti[p];
    for (int i = 0; i < n_candidate; ++i) {                      // np.random.uniform(xmin, xmax, n_candidate)
        const unsigned a = mt_next(mt, idx, P, p) >> 5, b = mt_next(mt, idx, P, p) >> 6;
        const double u = __dmul_rn(__dadd_rn(__dmul_rn((double)a, 67108864.0), (double)b), 1.0 / 9007199254740992.0);
        xc[i] = __dadd_rn(lo, __dmul_rn(range, u));
    }
    mti[p] = idx;
    // bq_c.filter_candidates (bq_c.pyx:622-650): merge close candidates until nothing changes, then drop those
    // that are close to an observation
    bool done = false;
    while (!done) {
        done = true;
        for (int i = 0; i < n_candidate; ++i) {
            if (isnan(xc[i])) continue;
            for (int j = i + 1; j < n_candidate; ++j) {
                if (isnan(xc[j])) continue;
                if (fabs(xc[i] - xc[j]) < thresh) {
                    xc[i] = (xc[i] + xc[j]) / 2.0;
                    xc[j] = nan("");
                    done = false;
                }
            }
        }
    }
    for (int j = 0; j < n; ++j) {
        const double v = xs[j];
        for (int i = 0; i < n_candidate; ++i)
            if (fabs(xc[i] - v) < thresh) xc[i] = nan("");       // NaN compares false
    }
    // np.sort(xc[~isnan]): insertion sort of at most NC_MAX survivors
    double out[NC_MAX];
    int m = 0;
    for (int i = 0; i < n_candidate; ++i) {
        const double v = xc[i];
        if (isnan(v)) continue;
        int k = m++;
        while (k > 0 && out[k - 1] > v) { out[k] = out[k - 1]; --k; }
        out[k] = v;
    }
    for (int i = 0; i < NC_MAX; ++i) x_c[(size_t)p * NC_MAX + i] = i < m ? out[i] : 0.0;
    nc[p] = m;
}

__global__ void draw_candidates_kernel(const double *__restrict__ x_s, const int *__restrict__ ns, int stride,
                                       const double *__restrict__ hyp, const double *__restrict__ prior,
                                       unsigned *__restrict__ mt, int *__restrict__ mti, int n_candidate,
                                       double *__restrict__ x_c, int *__restrict__ nc, int P) {
    draw_candidates_body<false>(x_s, ns, stride, hyp, nullptr, prior, mt, mti, n_candidate, x_c, nc, P);
}

__global__ void draw_candidates_wrapped_kernel(const double *__restrict__ x_s, const int *__restrict__ ns, int stride,
                                               const double *__restrict__ period, const double *__restrict__ prior,
                                               unsigned *__restrict__ mt, int *__restrict__ mti, int n_candidate,
                                               double *__restrict__ x_c, int *__restrict__ nc, int P) {
    draw_candidates_body<true>(x_s, ns, stride, nullptr, period, prior, mt, mti, n_candidate, x_c, nc, P);
}

cudaError_t launch_mt_seed(const unsigned *seeds, unsigned *mt, int *mti, int P, cudaStream_t s) {
    mt_seed_kernel<<<(P + 127) / 128, 128, 0, s>>>(seeds, mt, mti, P);
    return cudaGetLastError();
}

cudaError_t launch_add_observations(double *x_s, double *l_s, int *ns, int stride, const double *prior, const double *x_new,
                                    const double *l_new, int P, int *overflow, cudaStream_t s) {
    add_observations_kernel<<<(P + 127) / 128, 128, 0, s>>>(x_s, l_s, ns, stride, prior, x_new, l_new, P, overflow);
    return cudaGetLastError();
}

cudaError_t launch_draw_candidates(const double *x_s, const int *ns, int stride, const double *hyp, const double *prior,
                                   unsigned *mt, int *mti, int n_candidate, double *x_c, int *nc, int P, cudaStream_t s) {
    draw_candidates_kernel<<<(P + 127) / 128, 128, 0, s>>>(x_s, ns, stride, hyp, prior, mt, mti, n_candidate, x_c, nc, P);
    return cudaGetLastError();
}

cudaError_t launch_draw_candidates_wrapped(const double *x_s, const int *ns, int stride, const double *period, const double *prior,
                                           unsigned *mt, int *mti, int n_candidate, double *x_c, int *nc, int P, cudaStream_t s) {
    draw_candidates_wrapped_kernel<<<(P + 127) / 128, 128, 0, s>>>(x_s, ns, stride, period, prior, mt, mti, n_candidate, x_c, nc, P);
    return cudaGetLastError();
}

}  // namespace bqb
