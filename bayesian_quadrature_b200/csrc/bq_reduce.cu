// Reductions of choose_next / marginalize (bq.py:640-665): the mean over hyper-parameter
// samples of -esm (sequential in sample order, like numpy's mean(axis=0) over rows), the
// expected variance Zm^2 + Zv - esm (bq.py:374-377), and a deterministic (min, first index)
// reduction that shards combine across GPUs.
#include "bq_common.cuh"

namespace bqb {

__global__ void mean_neg_kernel(const double *__restrict__ esm, long long stride, int n_inst, long long na,
                                double *__restrict__ loss) {
    for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < na; p += (long long)gridDim.x * blockDim.x) {
        double s = 0;
        for (int b = 0; b < n_inst; ++b) s += -esm[(size_t)b * stride + p];   // pairwise-free: sample order
        loss[p] = s / n_inst;
    }
}

// acc[p] += -esm[0][p] - esm[1][p] - ... in row order, starting from acc[p]: walking a batch of hyper-parameter samples
// through a chunk-sized score buffer performs exactly the additions of mean_neg_kernel (and of numpy's mean(axis=0)), in the
// same order, without ever holding the [n_samples, na] matrix (819 MB at BASELINE configs[3]).
__global__ void sum_neg_accum_kernel(const double *__restrict__ esm, long long stride, int n_rows, long long na, double *__restrict__ acc) {
    for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < na; p += (long long)gridDim.x * blockDim.x) {
        double s = acc[p];
        for (int b = 0; b < n_rows; ++b) s += -esm[(size_t)b * stride + p];
        acc[p] = s;
    }
}

// Segmented form for many problems with S samples each: acc[g][p] += -esm[g*S][p] - esm[g*S+1][p] - ... in row order.  Per group
// these are the additions of sum_neg_accum_kernel, so one group reproduces it bit for bit and a problem's samples may arrive
// in chunks.  HBM-bound: every esm element is read once, acc is read and written once per launch.
__global__ void sum_neg_groups_kernel(const double *__restrict__ esm, long long stride, int n_groups, int group_size, long long na,
                                      double *__restrict__ acc, long long acc_stride) {
    for (int g = blockIdx.y; g < n_groups; g += gridDim.y) {
        const double *e = esm + (size_t)g * group_size * stride;
        double *a = acc + (size_t)g * acc_stride;
        for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < na; p += (long long)gridDim.x * blockDim.x) {
            double s = a[p];
#pragma unroll 4
            for (int r = 0; r < group_size; ++r) s += -e[(size_t)r * stride + p];
            a[p] = s;
        }
    }
}

__global__ void expected_var_kernel(const double *__restrict__ esm, long long na, double msm, double *__restrict__ out) {
    for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < na; p += (long long)gridDim.x * blockDim.x)
        out[p] = msm - esm[p];
}

__device__ __forceinline__ void better(double &v, long long &i, double v2, long long i2) {
    // NaN never wins; ties keep the smaller index (np.argmin semantics for finite data)
    if (v2 < v || (v2 == v && i2 < i)) { v = v2; i = i2; }
}

__global__ void argmin_kernel(const double *__restrict__ v, long long n, double *bv, long long *bi) {
    __shared__ double sv[32];
    __shared__ long long si[32];
    double best = INFINITY;
    long long idx = 0x7fffffffffffffffLL;
    for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x)
        better(best, idx, v[p], p);
    for (int o = 16; o > 0; o >>= 1) {
        const double v2 = __shfl_xor_sync(0xffffffffu, best, o);
        const long long i2 = __shfl_xor_sync(0xffffffffu, idx, o);
        better(best, idx, v2, i2);
    }
    if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = best; si[threadIdx.x >> 5] = idx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) better(best, idx, sv[w], si[w]);
        bv[blockIdx.x] = best;
        bi[blockIdx.x] = idx;
    }
}

__global__ void argmin_final_kernel(double *bv, long long *bi, int nblocks) {   // one warp
    double best = INFINITY;
    long long idx = 0x7fffffffffffffffLL;
    for (int b = threadIdx.x; b < nblocks; b += 32) better(best, idx, bv[b], bi[b]);
    for (int o = 16; o > 0; o >>= 1) {
        const double v2 = __shfl_xor_sync(0xffffffffu, best, o);
        const long long i2 = __shfl_xor_sync(0xffffffffu, idx, o);
        better(best, idx, v2, i2);
    }
    if (threadIdx.x == 0) { bv[0] = best; bi[0] = idx; }
}

// (min, global index as a double) pair for the cross-rank exchange: exact for indices < 2^53
__global__ void argmin_pair_kernel(const double *bv, const long long *bi, long long offset, double *pair) {
    if (threadIdx.x == 0) { pair[0] = bv[0]; pair[1] = (double)(bi[0] + offset); }
}

// One CTA per row: (min, first index) of every instance's score vector (C5: per-problem argmin)
__global__ void argmin_rows_kernel(const double *__restrict__ v, long long stride, long long n, double *mins, long long *idxs) {
    __shared__ double sv[32];
    __shared__ long long si[32];
    const double *row = v + (size_t)blockIdx.x * stride;
    double best = INFINITY;
    long long idx = 0x7fffffffffffffffLL;
    for (long long p = threadIdx.x; p < n; p += blockDim.x) better(best, idx, row[p], p);
    for (int o = 16; o > 0; o >>= 1) {
        const double v2 = __shfl_xor_sync(0xffffffffu, best, o);
        const long long i2 = __shfl_xor_sync(0xffffffffu, idx, o);
        better(best, idx, v2, i2);
    }
    if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = best; si[threadIdx.x >> 5] = idx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) better(best, idx, sv[w], si[w]);
        mins[blockIdx.x] = best;
        idxs[blockIdx.x] = idx;
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
    const long long n = (long long)n_inst * (H_COUNT + NC_MAX);
    const int blocks = (int)((n + 255) / 256 < 1184 ? (n + 255) / 256 : 1184);
    pack_info_kernel<<<blocks > 0 ? blocks : 1, 256, 0, s>>>(models, model_stride, off_lc, n_inst, out);
    return cudaGetLastError();
}

cudaError_t launch_argmin_rows(const double *v, long long stride, long long n, int rows, double *mins, long long *idxs,
                               cudaStream_t s) {
    argmin_rows_kernel<<<rows, 256, 0, s>>>(v, stride, n, mins, idxs);
    return cudaGetLastError();
}

cudaError_t launch_mean_neg(const double *esm, long long stride, int n_inst, long long na, double *loss, cudaStream_t s) {
    const int blocks = (int)((na + 255) / 256 < 2368 ? (na + 255) / 256 : 2368);
    mean_neg_kernel<<<blocks > 0 ? blocks : 1, 256, 0, s>>>(esm, stride, n_inst, na, loss);
    return cudaGetLastError();
}

cudaError_t launch_sum_neg_accum(const double *esm, long long stride, int n_rows, long long na, double *acc, cudaStream_t s) {
    const int blocks = (int)((na + 255) / 256 < 2368 ? (na + 255) / 256 : 2368);
    sum_neg_accum_kernel<<<blocks > 0 ? blocks : 1, 256, 0, s>>>(esm, stride, n_rows, na, acc);
    return cudaGetLastError();
}

cudaError_t launch_sum_neg_groups(const double *esm, long long stride, int n_groups, int group_size, long long na, double *acc,
                                  long long acc_stride, cudaStream_t s) {
    const int bx = (int)((na + 255) / 256 < 2368 ? (na + 255) / 256 : 2368);
    const int by = n_groups < 65535 ? n_groups : 65535;
    sum_neg_groups_kernel<<<dim3(bx > 0 ? bx : 1, by > 0 ? by : 1), 256, 0, s>>>(esm, stride, n_groups, group_size, na, acc, acc_stride);
    return cudaGetLastError();
}

cudaError_t launch_expected_var(const double *esm, long long na, double msm, double *out, cudaStream_t s) {
    const int blocks = (int)((na + 255) / 256 < 2368 ? (na + 255) / 256 : 2368);
    expected_var_kernel<<<blocks > 0 ? blocks : 1, 256, 0, s>>>(esm, na, msm, out);
    return cudaGetLastError();
}

cudaError_t launch_argmin(const double *v, long long n, double *bv, long long *bi, int sm_count, cudaStream_t s) {
    int blocks = (int)((n + 1023) / 1024);
    if (blocks > sm_count * 2) blocks = sm_count * 2;
    if (blocks > 4096) blocks = 4096;
    if (blocks < 1) blocks = 1;
    argmin_kernel<<<blocks, 256, 0, s>>>(v, n, bv, bi);
    argmin_final_kernel<<<1, 32, 0, s>>>(bv, bi, blocks);
    return cudaGetLastError();
}

// final step of the fused scoring epilogue: reduce the per-CTA partials and emit the (min, index + offset) pair
__global__ void argmin_partials_kernel(double *bv, long long *bi, int nblocks, long long offset, double *pair) {
    double best = INFINITY;
    long long idx = 0x7fffffffffffffffLL;
    for (int b = threadIdx.x; b < nblocks; b += 32) better(best, idx, bv[b], bi[b]);
    for (int o = 16; o > 0; o >>= 1) {
        const double v2 = __shfl_xor_sync(0xffffffffu, best, o);
        const long long i2 = __shfl_xor_sync(0xffffffffu, idx, o);
        better(best, idx, v2, i2);
    }
    if (threadIdx.x == 0) { pair[0] = best; pair[1] = (double)(idx + offset); }
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
    double best = INFINITY;
    long long idx = 0x7fffffffffffffffLL;
    for (int b = lane; b < nblocks; b += 32) better(best, idx, bv[b], bi[b]);
    for (int o = 16; o > 0; o >>= 1) {
        const double v2 = __shfl_xor_sync(0xffffffffu, best, o);
        const long long i2 = __shfl_xor_sync(0xffffffffu, idx, o);
        better(best, idx, v2, i2);
    }
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

cudaError_t launch_argmin_partials(double *bv, long long *bi, int nblocks, long long offset, double *pair, cudaStream_t s) {
    argmin_partials_kernel<<<1, 32, 0, s>>>(bv, bi, nblocks, offset, pair);
    return cudaGetLastError();
}

cudaError_t launch_argmin_pair(const double *bv, const long long *bi, long long offset, double *pair, cudaStream_t s) {
    argmin_pair_kernel<<<1, 32, 0, s>>>(bv, bi, offset, pair);
    return cudaGetLastError();
}

}  // namespace bqb
