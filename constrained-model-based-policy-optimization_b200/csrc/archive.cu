// Start-state sampling from the on-policy archive, on the device (SURVEY.md section 8f-1):
//   CPOBuffer.epoch_batch            buffers/cpobuffer.py:466-524   (uniform rows of every epoch)
//   CPOPolicy.compute_DKL            policies/cpo_policy.py:837-845 (network/ac_network.py:50-55)
//   CPOBuffer.boltz_dist             buffers/cpobuffer.py:385-396   (host: one number per epoch)
//   distributed_batch_from_archive   buffers/cpobuffer.py:413-463   (np.random.choice(N, B, p=dist))
// as called by algorithms/cmbpo.py:241-245 before every model-rollout batch.
//
// The archive columns stay resident in HBM.  An index sorted by epoch (stable counting sort, built
// once per archive update) turns "a uniform row of epoch e" into one Philox draw; the Boltzmann
// distribution is constant inside an epoch, so "a row with probability dist[row]" is "an epoch from
// the per-epoch CDF, then a uniform row of it".  Randomness is Philox4x32-10 keyed by (seed, draw
// id, sample index): reproducible, not the numpy stream (like the elite choice of the rollout).
#include "common.cuh"
#include "row_math.cuh"

namespace {

constexpr int IDX_BLOCK_ROWS = 2048;     // rows ranked by one warp, in order (stable)

// pass 1: per-block histogram of the bins (bin = epoch number, < 0 = empty row)
__global__ void archive_hist_kernel(const int32_t* __restrict__ epoch, int64_t N, int n_bins, int32_t* __restrict__ block_hist) {
    extern __shared__ int32_t sh_hist[];
    for (int i = threadIdx.x; i < n_bins; i += blockDim.x) sh_hist[i] = 0;
    __syncthreads();
    const int64_t r0 = (int64_t)blockIdx.x * IDX_BLOCK_ROWS;
    for (int i = threadIdx.x; i < IDX_BLOCK_ROWS && r0 + i < N; i += blockDim.x) {
        const int e = epoch[r0 + i];
        if (e >= 0 && e < n_bins) atomicAdd(&sh_hist[e], 1);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n_bins; i += blockDim.x) block_hist[(int64_t)i * gridDim.x + blockIdx.x] = sh_hist[i];
}

// pass 2: exclusive scan of the (bin-major, block-minor) histogram -> start of every (bin, block) run
// and the bin offsets.  One block; the table is small (n_bins x ceil(N / 2048)).
__global__ void archive_scan_kernel(int32_t* __restrict__ block_hist, int64_t n, int n_bins, int n_blocks,
                                    int64_t* __restrict__ bin_offsets) {
    __shared__ long long carry;
    __shared__ long long warp_sums[32];
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int64_t base = 0; base < n; base += blockDim.x) {
        const int64_t i = base + threadIdx.x;
        const long long v = i < n ? block_hist[i] : 0;
        long long x = v;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const long long y = __shfl_up_sync(0xffffffffu, x, off);
            if ((threadIdx.x & 31) >= off) x += y;
        }
        if ((threadIdx.x & 31) == 31) warp_sums[threadIdx.x >> 5] = x;
        __syncthreads();
        if (threadIdx.x < 32) {
            long long w = threadIdx.x < (blockDim.x >> 5) ? warp_sums[threadIdx.x] : 0;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const long long y = __shfl_up_sync(0xffffffffu, w, off);
                if (threadIdx.x >= off) w += y;
            }
            warp_sums[threadIdx.x] = w;
        }
        __syncthreads();
        const long long before = carry + ((threadIdx.x >> 5) ? warp_sums[(threadIdx.x >> 5) - 1] : 0) + x - v;
        if (i < n) {
            block_hist[i] = (int32_t)before;
            if (i % n_blocks == 0) bin_offsets[i / n_blocks] = before;
        }
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) carry += warp_sums[(blockDim.x >> 5) - 1];
        __syncthreads();
    }
    if (threadIdx.x == 0) bin_offsets[n_bins] = carry;
}

// pass 3: one warp per block of rows walks them in order; rows of equal bin in a group of 32 are
// ranked with match_any, so the scatter is STABLE (ascending row index inside a bin) and deterministic
__global__ void archive_scatter_kernel(const int32_t* __restrict__ epoch, int64_t N, int n_bins, int n_blocks,
                                       const int32_t* __restrict__ block_start, int32_t* __restrict__ sorted_idx) {
    extern __shared__ int32_t sh_next[];
    const int lane = threadIdx.x;
    for (int i = lane; i < n_bins; i += 32) sh_next[i] = block_start[(int64_t)i * n_blocks + blockIdx.x];
    __syncwarp();
    const int64_t r0 = (int64_t)blockIdx.x * IDX_BLOCK_ROWS;
    for (int i = 0; i < IDX_BLOCK_ROWS; i += 32) {
        const int64_t r = r0 + i + lane;
        int e = r < N ? epoch[r] : -1;
        if (e >= n_bins) e = -1;
        const unsigned same = __match_any_sync(0xffffffffu, e);
        const int rank = __popc(same & ((1u << lane) - 1u));
        int start = 0;
        if (e >= 0) start = sh_next[e];
        __syncwarp();
        if (e >= 0) {
            sorted_idx[start + rank] = (int32_t)r;
            if (rank == __popc(same) - 1) sh_next[e] = start + rank + 1;
        }
        __syncwarp();
    }
}

__device__ __forceinline__ uint32_t philox_u32(uint64_t seed, uint64_t draw, int64_t i, int stream) {
    uint32_t o[4];
    philox4x32_10((uint32_t)i, (uint32_t)((uint64_t)i >> 32), (uint32_t)draw, ((uint32_t)stream << 16) | (uint32_t)(draw >> 32),
                  (uint32_t)seed, (uint32_t)(seed >> 32), o);
    return o[0];
}
constexpr int RNG_STREAM_ARCHIVE = 7;

// uniform rows of given epochs: out[k * B + b] = a row of bin epochs[k]
__global__ void archive_sample_epochs_kernel(const int32_t* __restrict__ sorted_idx, const int64_t* __restrict__ bin_offsets,
                                             const int32_t* __restrict__ epochs, int n_ep, int64_t B, uint64_t seed,
                                             uint64_t draw, int32_t* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)n_ep * B) return;
    const int k = (int)(i / B);
    const int64_t lo = bin_offsets[epochs[k]], cnt = bin_offsets[epochs[k] + 1] - lo;
    const uint32_t u = philox_u32(seed, draw, i, RNG_STREAM_ARCHIVE);
    out[i] = cnt > 0 ? sorted_idx[lo + (int64_t)(((uint64_t)u * (uint64_t)cnt) >> 32)] : -1;
}

// rows with probability p(epoch) / count(epoch): epoch by inverse CDF, then a uniform row of it.  Samples
// [first, first + count) of a batch: sample i depends on (seed, draw, i) only, never on the batch size, so a
// shard writes exactly the rows the whole batch has at those positions
__global__ void archive_sample_boltz_kernel(const int32_t* __restrict__ sorted_idx, const int64_t* __restrict__ bin_offsets,
                                            const int32_t* __restrict__ epochs, const double* __restrict__ cdf, int n_ep,
                                            int64_t first, int64_t count, uint64_t seed, uint64_t draw,
                                            int32_t* __restrict__ out) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    const int64_t i = first + j;
    uint32_t o[4];
    philox4x32_10((uint32_t)i, (uint32_t)((uint64_t)i >> 32), (uint32_t)draw, ((uint32_t)(RNG_STREAM_ARCHIVE + 1) << 16) | (uint32_t)(draw >> 32),
                  (uint32_t)seed, (uint32_t)(seed >> 32), o);
    // 53-bit uniform in [0, 1), like numpy's random_sample that np.random.choice(p=...) searches its cdf with
    const double u = (double)(((uint64_t)(o[0] >> 5) << 26) | (uint64_t)(o[1] >> 6)) * (1.0 / 9007199254740992.0);
    int lo = 0, hi = n_ep - 1;              // first k with cdf[k] > u (searchsorted side='right'), clamped
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (cdf[mid] > u) hi = mid; else lo = mid + 1;
    }
    const int64_t start = bin_offsets[epochs[lo]], cnt = bin_offsets[epochs[lo] + 1] - start;
    out[j] = cnt > 0 ? sorted_idx[start + (int64_t)(((uint64_t)o[2] * (uint64_t)cnt) >> 32)] : -1;
}

__global__ void gather_rows_kernel(const float* __restrict__ src, int width, const int32_t* __restrict__ idx, int64_t n,
                                   float* __restrict__ dst) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * width) return;
    const int64_t r = i / width;
    const int c = (int)(i - r * width);
    const int32_t s = idx[r];
    dst[i] = s >= 0 ? src[(int64_t)s * width + c] : 0.f;
}

// mean over the B rows of every epoch of sum_a 0.5 (((mu1 - mu0)^2 + var0) / (var1 + 1e-8) - 1) + ls1 - ls0
// with (mu0, ls0) the CURRENT policy and (mu1, ls1) the archived one (ac_network.py:50-55,114).  The
// per-element expression is float32 in TF's op order; the sums run in float64.
__global__ void policy_kl_epochs_kernel(const float* __restrict__ cur_mu, const float* __restrict__ cur_log_std,
                                        const float* __restrict__ old_mu, const float* __restrict__ old_log_std,
                                        int64_t B, int A, double* __restrict__ sums) {
    const int k = blockIdx.y;
    double acc = 0.0;
    for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (int64_t)gridDim.x * blockDim.x) {
        const int64_t row = (int64_t)k * B + b;
        float s = 0.f;
        for (int a = 0; a < A; ++a) {
            const float ls0 = cur_log_std[a], ls1 = old_log_std[row * A + a];
            const float var0 = expf(__fmul_rn(2.f, ls0)), var1 = expf(__fmul_rn(2.f, ls1));
            const float d = __fsub_rn(old_mu[row * A + a], cur_mu[row * A + a]);
            const float q = __fdiv_rn(__fadd_rn(__fmul_rn(d, d), var0), __fadd_rn(var1, 1e-8f));
            const float pre = __fsub_rn(__fadd_rn(__fmul_rn(0.5f, __fsub_rn(q, 1.0f)), ls1), ls0);
            s = (a == 0) ? pre : __fadd_rn(s, pre);
        }
        acc += (double)s;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, off);
    __shared__ double sh[32];
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sh[w];
        atomicAdd(sums + k, t);
    }
}

}  // namespace

extern "C" int cmbpo_archive_index(cmbpo_ctx* ctx, const int32_t* epoch, int64_t N, int n_bins,
                                   int32_t* sorted_idx, int64_t* bin_offsets, int64_t* bin_offsets_host) {
    CMBPO_CHECK(ctx && epoch && sorted_idx && bin_offsets && bin_offsets_host, "null argument");
    CMBPO_CHECK(N >= 0 && N < (int64_t)1 << 31, "archive size %lld out of range", (long long)N);
    CMBPO_CHECK(n_bins > 0 && n_bins <= 8192, "epoch bins %d out of range (1..8192)", n_bins);
    const int n_blocks = max(1, cdiv(N, IDX_BLOCK_ROWS));
    int32_t* block_hist;
    const size_t tbl = (size_t)n_bins * n_blocks;
    if (cmbpo_ws_get(ctx, 5, tbl * sizeof(int32_t), (void**)&block_hist)) return 1;
    archive_hist_kernel<<<n_blocks, 256, n_bins * sizeof(int32_t), ctx->stream>>>(epoch, N, n_bins, block_hist);
    archive_scan_kernel<<<1, 1024, 0, ctx->stream>>>(block_hist, (int64_t)tbl, n_bins, n_blocks, bin_offsets);
    archive_scatter_kernel<<<n_blocks, 32, n_bins * sizeof(int32_t), ctx->stream>>>(epoch, N, n_bins, n_blocks, block_hist, sorted_idx);
    ctx->launches += 3;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(bin_offsets_host, bin_offsets, (size_t)(n_bins + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int cmbpo_archive_sample_epochs(cmbpo_ctx* ctx, const int32_t* sorted_idx, const int64_t* bin_offsets,
                                           const int32_t* epochs, int n_ep, int64_t B, uint64_t seed, uint64_t draw,
                                           int32_t* out_idx) {
    CMBPO_CHECK(ctx && sorted_idx && bin_offsets && epochs && out_idx, "null argument");
    const int64_t n = (int64_t)n_ep * B;
    if (n == 0) return 0;
    archive_sample_epochs_kernel<<<cdiv(n, 256), 256, 0, ctx->stream>>>(sorted_idx, bin_offsets, epochs, n_ep, B, seed, draw, out_idx);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int cmbpo_archive_sample_boltz(cmbpo_ctx* ctx, const int32_t* sorted_idx, const int64_t* bin_offsets,
                                          const int32_t* epochs, const double* cdf, int n_ep, int64_t B,
                                          uint64_t seed, uint64_t draw, int32_t* out_idx) {
    return cmbpo_archive_sample_boltz_range(ctx, sorted_idx, bin_offsets, epochs, cdf, n_ep, 0, B, seed, draw, out_idx);
}

extern "C" int cmbpo_archive_sample_boltz_range(cmbpo_ctx* ctx, const int32_t* sorted_idx, const int64_t* bin_offsets,
                                                const int32_t* epochs, const double* cdf, int n_ep, int64_t first,
                                                int64_t count, uint64_t seed, uint64_t draw, int32_t* out_idx) {
    // an empty shard may pass out_idx = NULL (torch's pointer of an empty tensor)
    CMBPO_CHECK(ctx && sorted_idx && bin_offsets && epochs && cdf && (out_idx || count == 0), "null argument");
    CMBPO_CHECK(n_ep > 0, "no epochs to sample from");
    CMBPO_CHECK(first >= 0 && count >= 0, "sample range [%lld, +%lld) out of range", (long long)first, (long long)count);
    if (count == 0) return 0;
    archive_sample_boltz_kernel<<<cdiv(count, 256), 256, 0, ctx->stream>>>(sorted_idx, bin_offsets, epochs, cdf, n_ep,
                                                                         first, count, seed, draw, out_idx);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int cmbpo_gather_rows(cmbpo_ctx* ctx, const float* src, int width, const int32_t* idx, int64_t n, float* dst) {
    CMBPO_CHECK(ctx && src && idx && dst && width > 0, "bad argument");
    if (n == 0) return 0;
    gather_rows_kernel<<<cdiv(n * width, 256), 256, 0, ctx->stream>>>(src, width, idx, n, dst);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int cmbpo_policy_kl_epochs(cmbpo_ctx* ctx, const float* cur_mu, const float* cur_log_std, const float* old_mu,
                                      const float* old_log_std, int n_ep, int64_t B, int A, double* kl_host) {
    CMBPO_CHECK(ctx && cur_mu && cur_log_std && old_mu && old_log_std && kl_host, "null argument");
    CMBPO_CHECK(n_ep > 0 && n_ep <= 65535 && B > 0 && A > 0, "bad shape");
    double* sums;
    if (cmbpo_ws_get(ctx, 6, (size_t)n_ep * sizeof(double), (void**)&sums)) return 1;
    CUDA_TRY(cudaMemsetAsync(sums, 0, (size_t)n_ep * sizeof(double), ctx->stream));
    dim3 grid(max(1, min(cdiv(B, 256), ctx->sm_count * 2)), n_ep);
    policy_kl_epochs_kernel<<<grid, 256, 0, ctx->stream>>>(cur_mu, cur_log_std, old_mu, old_log_std, B, A, sums);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(kl_host, sums, (size_t)n_ep * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    for (int k = 0; k < n_ep; ++k) kl_host[k] /= (double)B;      // tf.reduce_mean over the batch
    return 0;
}
