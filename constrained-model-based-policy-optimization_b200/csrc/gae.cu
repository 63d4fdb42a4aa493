// K3 / K4: GAE + cost-GAE reverse scans, advantage statistics / normalisation and the
// populated-mask compaction of ModelBuffer.get().
//
// Reference arithmetic (buffers/modelbuffer.py:163-179, buffers/cpobuffer.py:179-207,
// utilities/utils.py:186-188):
//     delta_t = fl32( fl32(r_t + fl32(gamma32 * v_{t+1})) - v_t ),  v_T = last_val
//     y_t     = fl64( delta_t + fl64(d * y_{t+1}) ),  d = gamma*lam in float64   (scipy lfilter, DF-II-T)
//     adv_t   = fl32(y_t);  ret_t = fl32(adv_t + v_t)
// HBM-bound: 16 B read + 16 B written per step.
#include "common.cuh"

namespace {

struct GaeK {
    float g32, cg32;     // float32(gamma), float32(cost_gamma): numpy casts the python scalar
    double d, cd;        // gamma*lam, cgamma*clam in float64
};

// one scan step, op order as documented above
__device__ __forceinline__ void gae_step(float r, float v, float vnext, float g32, double d, double& y,
                                         float& adv, float& ret) {
    float delta = __fsub_rn(__fadd_rn(r, __fmul_rn(g32, vnext)), v);
    y = __dadd_rn((double)delta, __dmul_rn(d, y));
    adv = (float)y;
    ret = __fadd_rn(adv, v);
}

// ---- STRICT, generic strides: one thread per path, direct global access -------------------
// Coalesced when path_stride == 1 (the time-major rollout buffers).
__global__ void gae_paths_strict_kernel(const float* __restrict__ rew, const float* __restrict__ val,
                                        const float* __restrict__ cost, const float* __restrict__ cval,
                                        int64_t n_paths, int max_len, int64_t ps, int64_t ts,
                                        const int32_t* __restrict__ length,
                                        const float* __restrict__ last_val,
                                        const float* __restrict__ last_cval, GaeK k,
                                        float* __restrict__ adv, float* __restrict__ ret,
                                        float* __restrict__ cadv, float* __restrict__ cret) {
    int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_paths) return;
    int len = length ? length[p] : max_len;
    if (len <= 0) return;
    double y = 0.0, cy = 0.0;
    float vn = last_val[p], cvn = last_cval[p];
    const int64_t base = p * ps;
    // The recurrence is sequential, the loads are not: the inputs of GB consecutive steps (4 x GB independent,
    // warp-coalesced loads) are fetched before the first of them is consumed.  One thread per path gives only
    // ~30 % occupancy at 100 k paths, so the bytes in flight have to come from each thread.
    constexpr int GB = 8;      // measured: 8 loads x 4 arrays in flight per thread; 16 (and 64-thread blocks) was slower
    for (int t0 = len - 1; t0 >= 0; t0 -= GB) {
        float r[GB], v[GB], c[GB], cv[GB];
#pragma unroll
        for (int j = 0; j < GB; ++j) {
            const int t = t0 - j;
            if (t >= 0) {
                const int64_t i = base + (int64_t)t * ts;
                r[j] = __ldg(rew + i); v[j] = __ldg(val + i); c[j] = __ldg(cost + i); cv[j] = __ldg(cval + i);
            }
        }
#pragma unroll
        for (int j = 0; j < GB; ++j) {
            const int t = t0 - j;
            if (t >= 0) {
                const int64_t i = base + (int64_t)t * ts;
                float a, rt, ca, crt;
                gae_step(r[j], v[j], vn, k.g32, k.d, y, a, rt);
                gae_step(c[j], cv[j], cvn, k.cg32, k.cd, cy, ca, crt);
                adv[i] = a; ret[i] = rt; cadv[i] = ca; cret[i] = crt;
                vn = v[j]; cvn = cv[j];
            }
        }
    }
}

// ---- WARP, flat CPOBuffer layout: one warp per segment, 32-element chunks walked from the end
// of the segment to its start; inside a chunk the recurrence y_t = x_t + d*y_{t+1} is a
// Hillis-Steele scan over lanes with powers of d (5 shuffle rounds, float64), the carry enters
// as d^(k+1)*carry.
__device__ __forceinline__ double shfl_down_f64(double x, int delta) {
    return __shfl_down_sync(0xffffffffu, x, delta);
}

__global__ void gae_segments_warp_kernel(const float* __restrict__ rew, const float* __restrict__ val,
                                         const float* __restrict__ cost, const float* __restrict__ cval,
                                         int64_t n_seg, const int64_t* __restrict__ seg_offsets,
                                         const float* __restrict__ last_val,
                                         const float* __restrict__ last_cval, GaeK k,
                                         float* __restrict__ adv, float* __restrict__ ret,
                                         float* __restrict__ cadv, float* __restrict__ cret) {
    const int lane = threadIdx.x & 31;
    const int64_t seg = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (seg >= n_seg) return;
    const int64_t base = seg_offsets[seg];
    const int len = (int)(seg_offsets[seg + 1] - base);
    if (len <= 0) return;
    // powers of d for the in-chunk scan
    double dp[5], cdp[5];
    dp[0] = k.d; cdp[0] = k.cd;
#pragma unroll
    for (int i = 1; i < 5; ++i) { dp[i] = dp[i - 1] * dp[i - 1]; cdp[i] = cdp[i - 1] * cdp[i - 1]; }
    const float lv = last_val[seg], lcv = last_cval[seg];
    double carry = 0.0, ccarry = 0.0;     // y at the first element of the chunk processed before (later in time)
    for (int hi = len; hi > 0; hi -= 32) {
        const int lo = max(hi - 32, 0);
        const int t = lo + lane;
        const bool ok = t < hi;
        double x = 0.0, cx = 0.0;
        float v = 0.f, cv = 0.f;
        const int64_t i = base + t;
        if (ok) {
            float r = rew[i], c = cost[i];
            v = val[i]; cv = cval[i];
            float vn = (t + 1 < len) ? val[i + 1] : lv;
            float cvn = (t + 1 < len) ? cval[i + 1] : lcv;
            x = (double)__fsub_rn(__fadd_rn(r, __fmul_rn(k.g32, vn)), v);
            cx = (double)__fsub_rn(__fadd_rn(c, __fmul_rn(k.cg32, cvn)), cv);
        }
        // in-chunk inclusive reverse scan
#pragma unroll
        for (int s = 0; s < 5; ++s) {
            const int off = 1 << s;
            double o = shfl_down_f64(x, off), co = shfl_down_f64(cx, off);
            if (lane + off < 32) { x = fma(dp[s], o, x); cx = fma(cdp[s], co, cx); }
        }
        // carry from the later chunk: element at position t sees d^(hi - t) * carry
        const int e = hi - t;                 // 1..32 for valid lanes
        if (ok && hi < len) {
            double w = 1.0, cw = 1.0;
#pragma unroll
            for (int s = 0; s < 6; ++s) if (e & (1 << s)) {
                w *= (s < 5) ? dp[s] : dp[4] * dp[4];
                cw *= (s < 5) ? cdp[s] : cdp[4] * cdp[4];
            }
            x = fma(w, carry, x); cx = fma(cw, ccarry, cx);
        }
        if (ok) {
            float a = (float)x, ca = (float)cx;
            adv[i] = a; ret[i] = __fadd_rn(a, v);
            cadv[i] = ca; cret[i] = __fadd_rn(ca, cv);
        }
        carry = __shfl_sync(0xffffffffu, x, 0);     // lane 0 holds t == lo
        ccarry = __shfl_sync(0xffffffffu, cx, 0);
    }
}

// ---- STRICT flat: one thread per segment (exact, uncoalesced for long segments) -----------
__global__ void gae_flat_strict_kernel(const float* __restrict__ rew, const float* __restrict__ val,
                                       const float* __restrict__ cost, const float* __restrict__ cval,
                                       int64_t n_seg, const int64_t* __restrict__ seg_offsets,
                                       const float* __restrict__ last_val,
                                       const float* __restrict__ last_cval, GaeK k,
                                       float* __restrict__ adv, float* __restrict__ ret,
                                       float* __restrict__ cadv, float* __restrict__ cret) {
    int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_seg) return;
    int64_t b = seg_offsets[s], e = seg_offsets[s + 1];
    double y = 0.0, cy = 0.0;
    float vn = last_val[s], cvn = last_cval[s];
    for (int64_t i = e - 1; i >= b; --i) {
        float r = rew[i], v = val[i], c = cost[i], cv = cval[i];
        float a, rt, ca, crt;
        gae_step(r, v, vn, k.g32, k.d, y, a, rt);
        gae_step(c, cv, cvn, k.cg32, k.cd, cy, ca, crt);
        adv[i] = a; ret[i] = rt; cadv[i] = ca; cret[i] = crt;
        vn = v; cvn = cv;
    }
}

// ---- statistics ---------------------------------------------------------------------------
// valid (p,t): t < length[p]; iteration space is the dense [max_len][n_paths] grid walked in
// memory order of the fastest stride.
__device__ __forceinline__ double block_sum(double v, double* sh) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) sh[w] = v;
    __syncthreads();
    double r = 0.0;
    if (w == 0) {
        r = (l < (blockDim.x >> 5)) ? sh[l] : 0.0;
        for (int o = 16; o > 0; o >>= 1) r += __shfl_down_sync(0xffffffffu, r, o);
    }
    __syncthreads();
    return r;
}

__global__ void stats_pass1_kernel(const float* __restrict__ adv, const float* __restrict__ cadv,
                                   const float* __restrict__ ret, const float* __restrict__ cret,
                                   int64_t n_paths, int max_len, int64_t ps, int64_t ts,
                                   const int32_t* __restrict__ length, double* __restrict__ partial) {
    __shared__ double sh[32];
    double n = 0, sa = 0, sc = 0, sr = 0, scr = 0;
    const int64_t total = n_paths * (int64_t)max_len;
    const bool path_fast = ps <= ts;   // which index is contiguous
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        int64_t p, t;
        if (path_fast) { t = i / n_paths; p = i - t * n_paths; } else { p = i / max_len; t = i - p * max_len; }
        int len = length ? length[p] : max_len;
        if (t < len) {
            int64_t j = p * ps + t * ts;
            n += 1.0; sa += adv[j]; sc += cadv[j]; sr += ret[j]; scr += cret[j];
        }
    }
    n = block_sum(n, sh); sa = block_sum(sa, sh); sc = block_sum(sc, sh);
    sr = block_sum(sr, sh); scr = block_sum(scr, sh);
    if (threadIdx.x == 0) {
        double* o = partial + (size_t)blockIdx.x * 8;
        o[0] = n; o[1] = sa; o[2] = sc; o[3] = sr; o[4] = scr; o[5] = 0; o[6] = 0; o[7] = 0;
    }
}

__global__ void stats_pass2_kernel(const float* __restrict__ adv, int64_t n_paths, int max_len,
                                   int64_t ps, int64_t ts, const int32_t* __restrict__ length,
                                   const double* __restrict__ sums, double* __restrict__ partial) {
    __shared__ double sh[32];
    double ss = 0;
    // mean = float32(sum) / float32(n) as mpi_tools.py:82-83, from the (all-reduced) sums of pass 1
    const float mean = (sums[0] > 0.0) ? __fdiv_rn((float)sums[1], (float)sums[0]) : 0.f;
    const int64_t total = n_paths * (int64_t)max_len;
    const bool path_fast = ps <= ts;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        int64_t p, t;
        if (path_fast) { t = i / n_paths; p = i - t * n_paths; } else { p = i / max_len; t = i - p * max_len; }
        int len = length ? length[p] : max_len;
        if (t < len) {
            float d = __fsub_rn(adv[p * ps + t * ts], mean);     // float32 (x - mean)**2, mpi_tools.py:85
            ss += (double)__fmul_rn(d, d);
        }
    }
    ss = block_sum(ss, sh);
    if (threadIdx.x == 0) partial[blockIdx.x] = ss;
}

// fixed-order final reduction -> deterministic for a fixed grid: thread t sums blocks t, t+256, ...
// in order, then a fixed shared-memory tree (one block; `width` columns handled one after the other)
__global__ void __launch_bounds__(256) stats_final_kernel(const double* __restrict__ partial, int n_blocks, int width,
                                                          int stride, double* __restrict__ out, int out_offset) {
    __shared__ double sh[256];
    for (int c = 0; c < width; ++c) {
        double s = 0;
        for (int b = threadIdx.x; b < n_blocks; b += 256) s += partial[(size_t)b * stride + c];
        sh[threadIdx.x] = s;
        __syncthreads();
        for (int off = 128; off > 0; off >>= 1) {
            if (threadIdx.x < off) sh[threadIdx.x] += sh[threadIdx.x + off];
            __syncthreads();
        }
        if (threadIdx.x == 0) out[out_offset + c] = sh[0];
        __syncthreads();
    }
}

__global__ void normalise_kernel(float* __restrict__ adv, float* __restrict__ cadv, int64_t n_paths,
                                 int max_len, int64_t ps, int64_t ts,
                                 const int32_t* __restrict__ length, const double* __restrict__ sums) {
    // sums = (n, sum adv, sum cadv, sum ret, sum cret, sum (adv-mean)^2), all-reduced
    if (!(sums[0] > 0.0)) return;
    const float n = (float)sums[0];
    const float mean = __fdiv_rn((float)sums[1], n);
    const float cmean = __fdiv_rn((float)sums[2], n);
    const float denom = __fadd_rn(__fsqrt_rn(__fdiv_rn((float)sums[5], n)), 1e-8f);     // mpi_tools.py:85-86, modelbuffer.py:199
    const int64_t total = n_paths * (int64_t)max_len;
    const bool path_fast = ps <= ts;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        int64_t p, t;
        if (path_fast) { t = i / n_paths; p = i - t * n_paths; } else { p = i / max_len; t = i - p * max_len; }
        int len = length ? length[p] : max_len;
        if (t < len) {
            int64_t j = p * ps + t * ts;
            adv[j] = __fdiv_rn(__fsub_rn(adv[j], mean), denom);   // modelbuffer.py:199
            cadv[j] = __fsub_rn(cadv[j], cmean);                  // modelbuffer.py:204
        }
    }
}

// ---- exclusive prefix sum of path lengths (3 small kernels) -------------------------------
constexpr int SCAN_THREADS = 256, SCAN_ITEMS = 16, SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__global__ void scan_tile_sums(const int32_t* __restrict__ len, int64_t B, int64_t* __restrict__ tile_sum) {
    __shared__ double sh[32];
    int64_t base = (int64_t)blockIdx.x * SCAN_TILE;
    double s = 0;
    for (int i = threadIdx.x; i < SCAN_TILE; i += SCAN_THREADS) {
        int64_t j = base + i;
        if (j < B) s += len[j];
    }
    s = block_sum(s, sh);
    if (threadIdx.x == 0) tile_sum[blockIdx.x] = (int64_t)s;
}

__global__ void scan_tile_offsets(int64_t* tile_sum, int n_tiles, int64_t* total_out) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        int64_t run = 0;
        for (int i = 0; i < n_tiles; ++i) { int64_t v = tile_sum[i]; tile_sum[i] = run; run += v; }
        *total_out = run;
    }
}

__global__ void scan_apply(const int32_t* __restrict__ len, int64_t B, const int64_t* __restrict__ tile_off,
                           int64_t* __restrict__ out) {
    __shared__ int64_t sh[SCAN_THREADS];
    int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
    int32_t v[SCAN_ITEMS];
    int64_t s = 0;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) { v[i] = (base + i < B) ? len[base + i] : 0; s += v[i]; }
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int o = 1; o < SCAN_THREADS; o <<= 1) {
        int64_t add = (threadIdx.x >= o) ? sh[threadIdx.x - o] : 0;
        __syncthreads();
        sh[threadIdx.x] += add;
        __syncthreads();
    }
    int64_t run = tile_off[blockIdx.x] + sh[threadIdx.x] - s;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) { if (base + i < B) out[base + i] = run; run += v[i]; }
}

// ---- buf[populated_mask] for a time-major field -------------------------------------------
__global__ void compact_kernel(const float* __restrict__ field, int64_t B, int T, int width,
                               const int32_t* __restrict__ length, const int64_t* __restrict__ row_off,
                               float* __restrict__ out) {
    const int64_t total = (int64_t)T * B * width;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        int w = (int)(i % width);
        int64_t pt = i / width;
        int64_t t = pt / B, p = pt - t * B;
        if (t < length[p]) out[(row_off[p] + t) * width + w] = field[i];
    }
}

__global__ void scatter_rows_kernel(float* __restrict__ dst, int64_t B, int width, int t,
                                    const int32_t* __restrict__ idx, const float* __restrict__ src,
                                    int64_t n) {
    const int64_t total = n * width;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        int64_t r = i / width;
        int w = (int)(i - r * width);
        dst[((int64_t)t * B + idx[r]) * width + w] = src[i];
    }
}

GaeK make_k(double gamma, double lam, double cgamma, double clam) {
    GaeK k;
    k.g32 = (float)gamma; k.cg32 = (float)cgamma;
    k.d = gamma * lam; k.cd = cgamma * clam;
    return k;
}

int grid_for(cmbpo_ctx* ctx, int64_t total, int threads) {
    int64_t want = (total + threads - 1) / threads;
    int64_t cap = (int64_t)ctx->sm_count * 8;
    return (int)(want < 1 ? 1 : (want > cap ? cap : want));
}

}  // namespace

extern "C" int cmbpo_gae_paths(cmbpo_ctx* ctx, const float* rew, const float* val, const float* cost,
                               const float* cval, int64_t n_paths, int max_len, int64_t path_stride,
                               int64_t time_stride, const int32_t* length, const float* last_val,
                               const float* last_cval, double gamma, double lam, double cgamma,
                               double clam, float* adv, float* ret, float* cadv, float* cret) {
    CMBPO_CHECK(ctx, "null context");
    if (n_paths <= 0 || max_len <= 0) return 0;
    GaeK k = make_k(gamma, lam, cgamma, clam);
    ProfScope prof(ctx, CMBPO_PROF_GAE);
    int threads = 128;
    int64_t blocks = (n_paths + threads - 1) / threads;
    gae_paths_strict_kernel<<<(unsigned)blocks, threads, 0, ctx->stream>>>(
        rew, val, cost, cval, n_paths, max_len, path_stride, time_stride, length, last_val,
        last_cval, k, adv, ret, cadv, cret);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int cmbpo_gae_flat(cmbpo_ctx* ctx, const float* rew, const float* val, const float* cost,
                              const float* cval, const int64_t* seg_offsets, int64_t n_seg,
                              const float* last_val, const float* last_cval, double gamma, double lam,
                              double cgamma, double clam, float* adv, float* ret, float* cadv,
                              float* cret, int scan_mode) {
    CMBPO_CHECK(ctx, "null context");
    if (n_seg <= 0) return 0;
    GaeK k = make_k(gamma, lam, cgamma, clam);
    ProfScope prof(ctx, CMBPO_PROF_GAE);
    int threads = 256;
    if (scan_mode == CMBPO_SCAN_WARP) {
        int64_t blocks = (n_seg * 32 + threads - 1) / threads;
        gae_segments_warp_kernel<<<(unsigned)blocks, threads, 0, ctx->stream>>>(
            rew, val, cost, cval, n_seg, seg_offsets, last_val, last_cval, k, adv, ret, cadv, cret);
    } else {
        int64_t blocks = (n_seg + 63) / 64;
        gae_flat_strict_kernel<<<(unsigned)blocks, 64, 0, ctx->stream>>>(
            rew, val, cost, cval, n_seg, seg_offsets, last_val, last_cval, k, adv, ret, cadv, cret);
    }
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int cmbpo_adv_stats_pass1(cmbpo_ctx* ctx, const float* adv, const float* cadv,
                                     const float* ret, const float* cret, int64_t n_paths, int max_len,
                                     int64_t path_stride, int64_t time_stride, const int32_t* length,
                                     double* sums_out) {
    CMBPO_CHECK(ctx, "null context");
    int threads = 256;
    int blocks = grid_for(ctx, n_paths * (int64_t)max_len, threads);
    double* partial;
    if (cmbpo_ws_get(ctx, 7, (size_t)blocks * 8 * sizeof(double), (void**)&partial)) return 1;
    stats_pass1_kernel<<<blocks, threads, 0, ctx->stream>>>(adv, cadv, ret, cret, n_paths, max_len,
                                                          path_stride, time_stride, length, partial);
    stats_final_kernel<<<1, 256, 0, ctx->stream>>>(partial, blocks, 8, 8, sums_out, 0);
    ctx->launches += 2;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int cmbpo_adv_stats_pass2(cmbpo_ctx* ctx, const float* adv, int64_t n_paths, int max_len,
                                     int64_t path_stride, int64_t time_stride, const int32_t* length,
                                     const double* sums, double* sums_out) {
    CMBPO_CHECK(ctx && sums && sums_out, "null argument");
    int threads = 256;
    int blocks = grid_for(ctx, n_paths * (int64_t)max_len, threads);
    double* partial;
    if (cmbpo_ws_get(ctx, 7, (size_t)blocks * 8 * sizeof(double), (void**)&partial)) return 1;
    stats_pass2_kernel<<<blocks, threads, 0, ctx->stream>>>(adv, n_paths, max_len, path_stride,
                                                          time_stride, length, sums, partial);
    stats_final_kernel<<<1, 256, 0, ctx->stream>>>(partial, blocks, 1, 1, sums_out, 5);
    ctx->launches += 2;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int cmbpo_adv_normalise(cmbpo_ctx* ctx, float* adv, float* cadv, int64_t n_paths,
                                   int max_len, int64_t path_stride, int64_t time_stride,
                                   const int32_t* length, const double* sums) {
    CMBPO_CHECK(ctx && sums, "null argument");
    int threads = 256;
    int blocks = grid_for(ctx, n_paths * (int64_t)max_len, threads);
    normalise_kernel<<<blocks, threads, 0, ctx->stream>>>(adv, cadv, n_paths, max_len, path_stride,
                                                         time_stride, length, sums);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int cmbpo_path_offsets(cmbpo_ctx* ctx, const int32_t* length, int64_t B,
                                  int64_t* row_offsets) {
    CMBPO_CHECK(ctx, "null context");
    int n_tiles = (int)((B + SCAN_TILE - 1) / SCAN_TILE);
    if (n_tiles < 1) n_tiles = 1;
    int64_t* tile_sum;
    if (cmbpo_ws_get(ctx, 6, (size_t)n_tiles * sizeof(int64_t), (void**)&tile_sum)) return 1;
    scan_tile_sums<<<n_tiles, SCAN_THREADS, 0, ctx->stream>>>(length, B, tile_sum);
    scan_tile_offsets<<<1, 32, 0, ctx->stream>>>(tile_sum, n_tiles, row_offsets + B);
    scan_apply<<<n_tiles, SCAN_THREADS, 0, ctx->stream>>>(length, B, tile_sum, row_offsets);
    ctx->launches += 3;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int cmbpo_compact_field(cmbpo_ctx* ctx, const float* field, int64_t B, int T, int width,
                                   const int32_t* length, const int64_t* row_offsets, float* out) {
    CMBPO_CHECK(ctx, "null context");
    int threads = 256;
    int blocks = grid_for(ctx, (int64_t)T * B * width, threads);
    compact_kernel<<<blocks, threads, 0, ctx->stream>>>(field, B, T, width, length, row_offsets, out);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int cmbpo_scatter_rows(cmbpo_ctx* ctx, float* dst, int64_t B, int width, int t,
                                  const int32_t* path_idx, const float* src, int64_t n) {
    CMBPO_CHECK(ctx, "null context");
    if (n <= 0) return 0;
    int blocks = grid_for(ctx, n * width, 256);
    scatter_rows_kernel<<<blocks, 256, 0, ctx->stream>>>(dst, B, width, t, path_idx, src, n);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}
