// Reductions of choose_next / marginalize (bq.py:640-665): the mean over hyper-parameter
// samples of -esm (sequential in sample order, like numpy's mean(axis=0) over rows), the
// expected variance Zm^2 + Zv - esm (bq.py:374-377), a deterministic (min, first index)
// reduction that shards combine across GPUs, and the reference's random pick among the points
// within np.isclose of the minimum (bq.py:664-665).
#include "bq_common.cuh"

namespace bqb {

// CTAs of 256 threads for a grid-stride loop over n elements: one element per thread, at most `cap` CTAs, at least one
static int grid_1d(long long n, long long cap = 2368) {
    const long long blocks = (n + 255) / 256 < cap ? (n + 255) / 256 : cap;
    return blocks > 0 ? (int)blocks : 1;
}

// Segmented sum for many problems with S samples each: acc[g][p] += -esm[g*S][p] - esm[g*S+1][p] - ... in row order,
// starting from acc[g][p].  Walking a batch of hyper-parameter samples through a chunk-sized score buffer performs exactly
// the additions of numpy's mean(axis=0), in the same order, without ever holding the [n_samples, na] matrix (819 MB at
// BASELINE configs[3]), and a problem's samples may arrive in chunks.  MEAN: one group that starts from 0 and ends with
// one division by the row count (the mean itself).  HBM-bound: every esm element is read once, acc is read and written
// once per launch.
template <bool MEAN>
__global__ void sum_neg_groups_kernel(const double *__restrict__ esm, long long stride, int n_groups, int group_size, long long na,
                                      double *__restrict__ acc, long long acc_stride) {
    // (groups inside the point loop, row loop unrolled by the compiler: it then issues each row's load ahead of the previous
    // row's addition, which measured fastest for all three entry points)
    for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < na; p += (long long)gridDim.x * blockDim.x) {
        for (int g = blockIdx.y; g < n_groups; g += gridDim.y) {
            const double *e = esm + (size_t)g * group_size * stride + p;
            double *a = acc + (size_t)g * acc_stride + p;
            double s = MEAN ? 0.0 : *a;
            for (int r = 0; r < group_size; ++r) s += -e[(size_t)r * stride];
            *a = MEAN ? s / group_size : s;
        }
    }
}

// Row-wise expected variance of instances [inst0, inst0 + n_rows): out[r][p] = (Zm^2 + Zv) - esm[r][p] with Zm / Zv read
// from each instance's model header on the device (so that a device-resident setup needs no host round trip).  The
// rounding steps are those of the host entry point (Zm * Zm + Zv on the host, then one subtraction) and of the fused
// epilogue of the scoring kernels, spelled out so that no FMA contraction can change the bits.  esm and out may alias.
__global__ void expected_var_rows_kernel(const double *models, long long model_stride, int inst0, int n_rows, const double *esm,
                                         long long esm_stride, long long na, double *out, long long out_stride) {
    for (int r = blockIdx.y; r < n_rows; r += gridDim.y) {
        const double *M = models + (size_t)(inst0 + r) * model_stride;
        const double msm = __dadd_rn(__dmul_rn(M[H_ZM], M[H_ZM]), M[H_ZV]);          // bq.py:374
        const double *e = esm + (size_t)r * esm_stride;
        double *o = out + (size_t)r * out_stride;
        // esm and out may alias, so the compiler keeps each load behind the store before it: eight loads are issued ahead
        // of their stores to keep enough of them in flight
        const long long G = (long long)gridDim.x * blockDim.x;
        long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x;
        for (; p + 7 * G < na; p += 8 * G) {
            double v[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) v[k] = e[p + k * G];
#pragma unroll
            for (int k = 0; k < 8; ++k) o[p + k * G] = __dsub_rn(msm, v[k]);
        }
        for (; p < na; p += G) o[p] = __dsub_rn(msm, e[p]);
    }
}

// ---- (min, first index) of double vectors
// The rule: NaN never wins, ties keep the smaller index (np.argmin semantics for finite data).  It selects the
// lexicographically smallest non-NaN (value, index) pair, so the result does not depend on the order of the reduction.
constexpr long long NO_INDEX = 0x7fffffffffffffffLL;

__device__ __forceinline__ void better(double &v, long long &i, double v2, long long i2) {
    if (v2 < v || (v2 == v && i2 < i)) { v = v2; i = i2; }
}

__device__ __forceinline__ void warp_argmin(double &v, long long &i) {            // every lane ends with the warp's pair
    for (int o = 16; o > 0; o >>= 1) {
        const double v2 = __shfl_xor_sync(0xffffffffu, v, o);
        const long long i2 = __shfl_xor_sync(0xffffffffu, i, o);
        better(v, i, v2, i2);
    }
}

__device__ __forceinline__ void block_argmin(double &v, long long &i) {           // thread 0 ends with the CTA's pair
    __shared__ double sv[32];
    __shared__ long long si[32];
    warp_argmin(v, i);
    if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = v; si[threadIdx.x >> 5] = i; }
    __syncthreads();
    if (threadIdx.x == 0)
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) better(v, i, sv[w], si[w]);
}

// One warp: the pair of nblocks per-CTA partials (argmin_kernel's or the scoring epilogue's), in every lane
__device__ __forceinline__ void partials_argmin(const double *bv, const long long *bi, int nblocks, double &v, long long &i) {
    v = INFINITY;
    i = NO_INDEX;
    for (int b = threadIdx.x; b < nblocks; b += 32) better(v, i, bv[b], bi[b]);
    warp_argmin(v, i);
}

__global__ void argmin_kernel(const double *__restrict__ v, long long n, double *bv, long long *bi) {
    double best = INFINITY;
    long long idx = NO_INDEX;
    for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x)
        better(best, idx, v[p], p);
    block_argmin(best, idx);
    if (threadIdx.x == 0) { bv[blockIdx.x] = best; bi[blockIdx.x] = idx; }
}

// One CTA per row: (min, first index) of every instance's score vector (C5: per-problem argmin)
__global__ void argmin_rows_kernel(const double *__restrict__ v, long long stride, long long n, double *mins, long long *idxs) {
    const double *row = v + (size_t)blockIdx.x * stride;
    double best = INFINITY;
    long long idx = NO_INDEX;
    for (long long p = threadIdx.x; p < n; p += blockDim.x) better(best, idx, row[p], p);
    block_argmin(best, idx);
    if (threadIdx.x == 0) { mins[blockIdx.x] = best; idxs[blockIdx.x] = idx; }
}

// numpy's isclose(v, m) with its default tolerances, argument order included (bq.py:664: isclose(loss, best)):
// |v - m| <= 1e-8 + 1e-5 * |m| for a finite m, or v == m -- equal infinities are close, a finite value is never close to an
// infinite one, NaN is close to nothing.  Each rounding step is spelled out so that no FMA contraction moves the boundary.
__device__ __forceinline__ bool isclose_np(double v, double m) {
    return (fabs(__dsub_rn(v, m)) <= __dadd_rn(1e-8, __dmul_rn(1e-5, fabs(m))) && isfinite(m)) || v == m;
}

// One CTA per row: the reference's random tie-break (bq.py:664-665, np.random.choice over the points isclose to the
// minimum).  Pass 1 counts the c points of row r close to mins[r]; pass 2 finds the k-th of them in ascending index order,
// k = min(floor(u[r] * c), c - 1), a tile of blockDim points at a time (a barrier count per tile, a ballot prefix inside the
// tile that holds it).  The second pass stops at that tile and mostly re-reads what pass 1 left in L2.  A row with no close
// point (all NaN) gets NO_INDEX, as argmin_rows_kernel gives it.
__global__ void argmin_ties_rows_kernel(const double *__restrict__ v, long long stride, long long n, const double *__restrict__ mins,
                                        const double *__restrict__ u, long long *idxs, long long *counts) {
    __shared__ long long s_count[32];
    __shared__ int s_warp[32];
    const double *row = v + (size_t)blockIdx.x * stride;
    const double m = mins[blockIdx.x];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    long long c = 0;
    for (long long p = threadIdx.x; p < n; p += blockDim.x) c += isclose_np(row[p], m);
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (lane == 0) s_count[warp] = c;
    __syncthreads();
    c = 0;
    for (int w = 0; w < nwarps; ++w) c += s_count[w];          // every thread: the row's count
    if (c == 0) {
        if (threadIdx.x == 0) {
            idxs[blockIdx.x] = NO_INDEX;
            if (counts) counts[blockIdx.x] = 0;
        }
        return;
    }
    long long k = (long long)__dmul_rn(u[blockIdx.x], (double)c);    // floor: the product is non-negative
    if (k > c - 1) k = c - 1;
    long long seen = 0;                                        // close points in the tiles before this one
    for (long long t = 0; t < n; t += blockDim.x) {
        const long long p = t + threadIdx.x;
        const bool hit = p < n && isclose_np(row[p], m);
        const unsigned ball = __ballot_sync(0xffffffffu, hit);
        if (lane == 0) s_warp[warp] = __popc(ball);
        // (the barrier also orders the s_warp stores before their reads; those happen only in the tile that ends the loop)
        const int in_tile = __syncthreads_count(hit);
        if (seen + in_tile > k) {                              // the k-th close point lies in this tile
            if (hit) {
                long long rank = seen + __popc(ball & ((1u << lane) - 1u));
                for (int w = 0; w < warp; ++w) rank += s_warp[w];
                if (rank == k) idxs[blockIdx.x] = p;
            }
            break;
        }
        seen += in_tile;
    }
    if (threadIdx.x == 0 && counts) counts[blockIdx.x] = c;
}

// One warp: reduces the per-CTA partials into bv[0] / bi[0] and, when `pair` is given, emits the (min, global index as a
// double) pair for the cross-rank exchange: exact for indices < 2^53
__global__ void argmin_partials_kernel(double *bv, long long *bi, int nblocks, long long offset, double *pair) {
    double best;
    long long idx;
    partials_argmin(bv, bi, nblocks, best, idx);
    if (threadIdx.x == 0) {
        bv[0] = best;
        bi[0] = idx;
        if (pair) { pair[0] = best; pair[1] = (double)(idx + offset); }
    }
}

// Per-instance setup results (header + l_c row) gathered into one contiguous [n_inst][H_COUNT + NC_MAX] array, so that they
// reach the host in ONE copy (a strided cudaMemcpy2D of 16384 rows of 256 B costs a DMA descriptor per row)
__global__ void pack_info_kernel(const double *__restrict__ models, long long model_stride, int off_lc, int n_inst, double *__restrict__ out) {
    constexpr int W = H_COUNT + NC_MAX;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < (long long)n_inst * W; e += (long long)gridDim.x * blockDim.x) {
        const long long i = e / W;
        const int j = (int)(e - i * W);
        out[e] = models[i * model_stride + (j < H_COUNT ? j : off_lc + (j - H_COUNT))];
    }
}
cudaError_t launch_pack_info(const double *models, long long model_stride, int off_lc, int n_inst, double *out, cudaStream_t s) {
    pack_info_kernel<<<grid_1d((long long)n_inst * (H_COUNT + NC_MAX), 1184), 256, 0, s>>>(models, model_stride, off_lc, n_inst, out);
    return cudaGetLastError();
}

cudaError_t launch_argmin_rows(const double *v, long long stride, long long n, int rows, double *mins, long long *idxs,
                               cudaStream_t s) {
    argmin_rows_kernel<<<rows, 256, 0, s>>>(v, stride, n, mins, idxs);
    return cudaGetLastError();
}

cudaError_t launch_argmin_ties_rows(const double *v, long long stride, long long n, int rows, const double *mins, const double *u,
                                    long long *idxs, long long *counts, cudaStream_t s) {
    argmin_ties_rows_kernel<<<rows, 256, 0, s>>>(v, stride, n, mins, u, idxs, counts);
    return cudaGetLastError();
}

// mean = false: acc[g] += the negated rows of group g; mean = true: acc = the mean of the negated rows of one group
cudaError_t launch_sum_neg_groups(const double *esm, long long stride, int n_groups, int group_size, long long na, double *acc,
                                  long long acc_stride, bool mean, cudaStream_t s) {
    const dim3 grid(grid_1d(na), n_groups < 1 ? 1 : n_groups < 65535 ? n_groups : 65535);
    if (mean)
        sum_neg_groups_kernel<true><<<grid, 256, 0, s>>>(esm, stride, n_groups, group_size, na, acc, acc_stride);
    else
        sum_neg_groups_kernel<false><<<grid, 256, 0, s>>>(esm, stride, n_groups, group_size, na, acc, acc_stride);
    return cudaGetLastError();
}

cudaError_t launch_expected_var_rows(const double *models, long long model_stride, int inst0, int n_rows, const double *esm,
                                     long long esm_stride, long long na, double *out, long long out_stride, cudaStream_t s) {
    const dim3 grid(grid_1d(na), n_rows < 1 ? 1 : n_rows < 65535 ? n_rows : 65535);
    expected_var_rows_kernel<<<grid, 256, 0, s>>>(models, model_stride, inst0, n_rows, esm, esm_stride, na, out, out_stride);
    return cudaGetLastError();
}

cudaError_t launch_argmin_partials(double *bv, long long *bi, int nblocks, long long offset, double *pair, cudaStream_t s) {
    argmin_partials_kernel<<<1, 32, 0, s>>>(bv, bi, nblocks, offset, pair);
    return cudaGetLastError();
}

// (min, first index) of v [n] into bv[0] / bi[0] (bv / bi hold the per-CTA partials first), and into pair when given
cudaError_t launch_argmin(const double *v, long long n, double *bv, long long *bi, int sm_count, long long offset, double *pair,
                          cudaStream_t s) {
    int blocks = (int)((n + 1023) / 1024);
    if (blocks > sm_count * 2) blocks = sm_count * 2;
    if (blocks > 4096) blocks = 4096;
    if (blocks < 1) blocks = 1;
    argmin_kernel<<<blocks, 256, 0, s>>>(v, n, bv, bi);
    return launch_argmin_partials(bv, bi, blocks, offset, pair, s);
}

// Fused "reduce + exchange" of choose_next over a sharded query vector (bq.py:663 across ranks): the one warp that
// reduces this rank's per-CTA partials stores its (min, first global index) pair straight into every rank's exchange
// buffer over NVLink (peer-mapped symmetric memory, slot [parity][writer rank]), flags it with the step number, waits for
// the other ranks' flags in its OWN buffer, and reduces the W pairs -- one small kernel instead of a reduction kernel, an
// NCCL all-gather and a device-to-host copy.  Two slot sets alternate with the step parity: a rank can be at most one
// step ahead of the slowest one (it needs that rank's flag of the current step), so a slot is never overwritten before
// it was read.  The spin is bounded; on time-out out[2] = 1.  `out` may be page-locked host memory.
struct PeerSlots {
    double *slot[16];
};
__global__ void argmin_exchange_kernel(const double *bv, const long long *bi, int nblocks, long long offset, long long cyc_block,
                                       PeerSlots peers, int world, int rank, unsigned long long seq, double *out) {
    const int lane = threadIdx.x;
    double best;
    long long idx;
    partials_argmin(bv, bi, nblocks, best, idx);
    const int par = (int)(seq & 1ull);
    const double tag = (double)seq;
    if (lane < world) {                                   // lane r publishes to rank r
        volatile double *dst = peers.slot[lane] + ((size_t)par * world + rank) * 4;
        dst[0] = best;
        // global index of this rank's local index: contiguous shard (offset) or block-cyclic shards of cyc_block points
        const long long g = cyc_block > 0 ? ((idx / cyc_block) * world + rank) * cyc_block + idx % cyc_block : idx + offset;
        dst[1] = (double)g;
        __threadfence_system();
        dst[2] = tag;
    }
    double v = INFINITY;
    long long gi = 0x7fffffffffffffffLL;
    int timed_out = 0;
    if (lane < world) {                                   // lane r collects rank r's pair
        volatile double *src = peers.slot[rank] + ((size_t)par * world + lane) * 4;
        long long spins = 0;
        while (src[2] != tag) {
            if (++spins > (1LL << 24)) { timed_out = 1; break; }
        }
        __threadfence_system();
        v = src[0];
        gi = (long long)src[1];
        if (v != v) v = INFINITY;                         // NaN never wins (np.nanargmin-free semantics of dist.combine_argmin)
    }
    for (int o = 16; o > 0; o >>= 1) {
        const double v2 = __shfl_xor_sync(0xffffffffu, v, o);
        const long long i2 = __shfl_xor_sync(0xffffffffu, gi, o);
        better(v, gi, v2, i2);
        timed_out |= __shfl_xor_sync(0xffffffffu, timed_out, o);
    }
    if (lane == 0) {
        out[0] = v;
        out[1] = (double)gi;
        out[2] = (double)timed_out;
        __threadfence_system();
        out[3] = tag;
    }
}

cudaError_t launch_argmin_exchange(const double *bv, const long long *bi, int nblocks, long long offset, long long cyc_block,
                                   void *const *peer_slots, int world, int rank, unsigned long long seq, double *out, cudaStream_t s) {
    if (world < 1 || world > 16 || rank < 0 || rank >= world) return cudaErrorInvalidValue;
    PeerSlots p;
    for (int r = 0; r < 16; ++r) p.slot[r] = r < world ? (double *)peer_slots[r] : nullptr;
    argmin_exchange_kernel<<<1, 32, 0, s>>>(bv, bi, nblocks, offset, cyc_block, p, world, rank, seq, out);
    return cudaGetLastError();
}

}  // namespace bqb
