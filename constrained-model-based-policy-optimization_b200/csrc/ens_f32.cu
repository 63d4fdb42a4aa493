// fp32 CUDA-core ensemble MLP chain.  This is the variant that isolates LOGIC from PRECISION:
// same data flow as the tcgen05 path, plain float32 FMA accumulation.
//
// Replaces FC.compute_output_tensor (models/pens/fc.py:74-95) applied layer by layer by
// PE._compile_outputs (models/pens/pe.py:804-812) with the input scaler of
// models/pens/utils.py:156 fused into the first layer's operand load.
#include "common.cuh"

namespace {

__device__ __forceinline__ float apply_act(int act, float x) {
    switch (act) {
        case CMBPO_ACT_SWISH: return __fmul_rn(x, __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-x))));  // fc.py:19
        case CMBPO_ACT_TANH: return tanhf(x);
        case CMBPO_ACT_RELU: return fmaxf(x, 0.0f);
        case CMBPO_ACT_SIGMOID: return __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-x)));
        default: return x;
    }
}

constexpr int BM = 64, BN = 64, BK = 16, TM = 4, TN = 4;   // 256 threads, 4x4 outputs each

// Y[e, n, m] = act( sum_k Xs[e, n, k] * W[e, k, m] + b[e, m] ),  Xs = (X - mu)/sigma if scaled
__global__ void __launch_bounds__(256)
ens_layer_f32_kernel(const float* __restrict__ X, int64_t x_member_stride, int ldx,
                     const float* __restrict__ W, const float* __restrict__ b,
                     float* __restrict__ Y, int64_t y_member_stride, int64_t N, int K, int M, int act,
                     const float* __restrict__ mu_in, const float* __restrict__ sig_in) {
    __shared__ float As[BK][BM + 4];
    __shared__ float Bs[BK][BN + 4];
    const int e = blockIdx.z;
    const int64_t row0 = (int64_t)blockIdx.y * BM;
    const int col0 = blockIdx.x * BN;
    const float* Xe = X + (int64_t)e * x_member_stride;
    const float* We = W + (int64_t)e * K * M;
    const int tid = threadIdx.x;
    const int tx = tid % (BN / TN), ty = tid / (BN / TN);
    float acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

    for (int k0 = 0; k0 < K; k0 += BK) {
        // A tile: BM x BK, 1024 elements, 4 per thread
#pragma unroll
        for (int it = 0; it < (BM * BK) / 256; ++it) {
            int idx = tid + it * 256;
            int r = idx / BK, kk = idx % BK;
            int64_t gr = row0 + r;
            int gk = k0 + kk;
            float v = 0.f;
            if (gr < N && gk < K) {
                v = Xe[gr * ldx + gk];
                if (mu_in) v = __fdiv_rn(__fsub_rn(v, mu_in[gk]), sig_in[gk]);   // pens/utils.py:156
            }
            As[kk][r] = v;
        }
#pragma unroll
        for (int it = 0; it < (BK * BN) / 256; ++it) {
            int idx = tid + it * 256;
            int kk = idx / BN, c = idx % BN;
            int gk = k0 + kk, gc = col0 + c;
            Bs[kk][c] = (gk < K && gc < M) ? We[(int64_t)gk * M + gc] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            float a[TM], bb[TN];
#pragma unroll
            for (int i = 0; i < TM; ++i) a[i] = As[kk][ty * TM + i];
#pragma unroll
            for (int j = 0; j < TN; ++j) bb[j] = Bs[kk][tx * TN + j];
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
        }
        __syncthreads();
    }
    float* Ye = Y + (int64_t)e * y_member_stride;
    const float* be = b + (int64_t)e * M;
#pragma unroll
    for (int i = 0; i < TM; ++i) {
        int64_t gr = row0 + ty * TM + i;
        if (gr >= N) continue;
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            int gc = col0 + tx * TN + j;
            if (gc < M) Ye[gr * M + gc] = apply_act(act, __fadd_rn(acc[i][j], be[gc]));
        }
    }
}

// raw [E,N,2D] (or [E,N,D]) -> mean/var [E,N,D]   (pe.py:815-833, pens/utils.py:167,187)
__global__ void ens_head_kernel(const float* __restrict__ raw, int E, int64_t N, int D, int prob,
                                const float* __restrict__ mu_out, const float* __restrict__ sig_out,
                                const float* __restrict__ l2s_out, float* __restrict__ mean,
                                float* __restrict__ var) {
    const int64_t total = (int64_t)E * N * D;
    const int W = prob ? 2 * D : D;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        int d = (int)(i % D);
        int64_t en = i / D;
        float m = raw[en * W + d];
        if (mu_out) m = __fadd_rn(__fmul_rn(sig_out[d], m), mu_out[d]);
        mean[i] = m;
        if (prob && var) {
            float lv = raw[en * W + D + d];
            if (mu_out) lv = __fadd_rn(l2s_out[d], lv);
            var[i] = expf(lv);
        }
    }
}

// PE.predict: mean over members, var = mean var + var of means (pe.py:326-330, 343)
__global__ void ens_predict_mean_kernel(const float* __restrict__ raw, int E, int64_t N, int D, int prob,
                                        const float* __restrict__ mu_out,
                                        const float* __restrict__ sig_out,
                                        const float* __restrict__ l2s_out, float* __restrict__ mean,
                                        float* __restrict__ var) {
    const int64_t total = N * D;
    const int W = prob ? 2 * D : D;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        int d = (int)(i % D);
        int64_t n = i / D;
        float ms[CMBPO_MAX_E];
        float s = 0.f, sv = 0.f;
        for (int e = 0; e < E; ++e) {
            float m = raw[((int64_t)e * N + n) * W + d];
            if (mu_out) m = __fadd_rn(__fmul_rn(sig_out[d], m), mu_out[d]);
            ms[e] = m;
            s = (e == 0) ? m : __fadd_rn(s, m);
            if (prob) {
                float lv = raw[((int64_t)e * N + n) * W + D + d];
                if (mu_out) lv = __fadd_rn(l2s_out[d], lv);
                float v = expf(lv);
                sv = (e == 0) ? v : __fadd_rn(sv, v);
            }
        }
        float mbar = __fdiv_rn(s, (float)E);
        mean[i] = mbar;
        if (prob && var) {
            float q = 0.f;
            for (int e = 0; e < E; ++e) {
                float dd = __fsub_rn(ms[e], mbar);
                float d2 = __fmul_rn(dd, dd);
                q = (e == 0) ? d2 : __fadd_rn(q, d2);
            }
            var[i] = __fadd_rn(__fdiv_rn(sv, (float)E), __fdiv_rn(q, (float)E));
        }
    }
}

}  // namespace

// X [N,in] or [E,N,in] -> raw last-layer output [E,N,dims[L]].  Rows are processed in chunks so
// the two ping-pong activation scratch buffers stay small ([E, chunk, width]).
int ens_forward_f32(cmbpo_ctx* ctx, const Net& net, const float* x, int64_t N, bool x_is_3d,
                    float* out_raw) {
    CMBPO_CHECK(net.loaded, "network not loaded");
    if (N <= 0) return 0;
    const int64_t CH = 32768;
    int maxw = 0;
    for (int l = 1; l < net.n_layers; ++l) maxw = max(maxw, net.dims[l]);
    float *h0 = nullptr, *h1 = nullptr;
    const int64_t ch_rows = min(CH, N);
    if (net.n_layers > 1) {
        size_t bytes = (size_t)net.E * ch_rows * maxw * sizeof(float);
        if (cmbpo_ws_get(ctx, 0, bytes, (void**)&h0)) return 1;
        if (net.n_layers > 2 && cmbpo_ws_get(ctx, 1, bytes, (void**)&h1)) return 1;
    }
    const int Mlast = net.dims[net.n_layers];
    for (int64_t c0 = 0; c0 < N; c0 += CH) {
        const int64_t rows = min(CH, N - c0);
        const float* in = x + c0 * net.dims[0];
        int64_t in_stride = x_is_3d ? N * (int64_t)net.dims[0] : 0;
        for (int l = 0; l < net.n_layers; ++l) {
            const int K = net.dims[l], M = net.dims[l + 1];
            const bool last = (l == net.n_layers - 1);
            float* out = last ? out_raw + c0 * Mlast : ((l & 1) ? h1 : h0);
            const int64_t out_stride = last ? N * (int64_t)Mlast : rows * (int64_t)M;
            dim3 grid(cdiv(M, BN), cdiv(rows, BM), net.E);
            const bool scale = (l == 0) && net.has_in;
            ens_layer_f32_kernel<<<grid, 256, 0, ctx->stream>>>(
                in, in_stride, K, net.W[l], net.b[l], out, out_stride, rows, K, M, net.acts[l],
                scale ? net.mu_in : nullptr, scale ? net.sig_in : nullptr);
            ctx->launches++;
            in = out;
            in_stride = out_stride;
        }
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int ens_forward(cmbpo_ctx* ctx, Net& net, const float* x, int64_t N, bool x_is_3d, float* out_raw,
                int precision, const int64_t* n_dev) {
    ProfScope prof(ctx, (&net == &ctx->nets[CMBPO_NET_DYN]) ? CMBPO_PROF_DYN : -1);
    if (precision == CMBPO_PREC_FP32) return ens_forward_f32(ctx, net, x, N, x_is_3d, out_raw);   // all N rows
    CMBPO_CHECK(!x_is_3d, "tcgen05 path takes 2-D inputs only");
    CMBPO_CHECK(ens_tc_supported(net),
                "tcgen05 path needs 2 hidden layers of equal width <= 512 (<= 64 inputs, <= 128 outputs, <= 96 above width 256) or 3-4 hidden "
                "layers of equal width <= 256 (<= 64 inputs, <= 128 outputs), swish or tanh; use precision fp32 for this network");
    return ens_forward_tc(ctx, net, x, N, out_raw, precision, n_dev);
}

static int raw_out(cmbpo_ctx* ctx, Net& net, int64_t N, float** raw) {
    size_t bytes = (size_t)net.E * N * net.dims[net.n_layers] * sizeof(float);
    return cmbpo_ws_get(ctx, 2, bytes, (void**)raw);
}

extern "C" int cmbpo_ens_predict(cmbpo_ctx* ctx, int which, const float* x, int64_t N, int x_is_3d,
                                 float* mean, float* var, int precision) {
    CMBPO_CHECK(ctx && which >= 0 && which < CMBPO_NET_COUNT, "bad arguments");
    Net& net = ctx->nets[which];
    CMBPO_CHECK(net.loaded, "network %d not loaded", which);
    if (N <= 0) return 0;
    float* raw;
    if (raw_out(ctx, net, N, &raw)) return 1;
    if (ens_forward(ctx, net, x, N, x_is_3d != 0, raw, precision)) return 1;
    int64_t total = (int64_t)net.E * N * net.D;
    int blocks = (int)min((int64_t)ctx->sm_count * 8, (total + 255) / 256);
    ens_head_kernel<<<blocks, 256, 0, ctx->stream>>>(raw, net.E, N, net.D, net.probabilistic,
                                                    net.has_out ? net.mu_out : nullptr, net.sig_out,
                                                    net.l2s_out, mean, var);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int cmbpo_ens_predict_mean(cmbpo_ctx* ctx, int which, const float* x, int64_t N, float* mean,
                                      float* var, int precision) {
    CMBPO_CHECK(ctx && which >= 0 && which < CMBPO_NET_COUNT, "bad arguments");
    Net& net = ctx->nets[which];
    CMBPO_CHECK(net.loaded, "network %d not loaded", which);
    CMBPO_CHECK(net.E <= CMBPO_MAX_E, "ensemble too large");
    if (N <= 0) return 0;
    float* raw;
    if (raw_out(ctx, net, N, &raw)) return 1;
    if (ens_forward(ctx, net, x, N, false, raw, precision)) return 1;
    int64_t total = N * net.D;
    int blocks = (int)min((int64_t)ctx->sm_count * 8, (total + 255) / 256);
    ens_predict_mean_kernel<<<blocks, 256, 0, ctx->stream>>>(
        raw, net.E, N, net.D, net.probabilistic, net.has_out ? net.mu_out : nullptr, net.sig_out,
        net.l2s_out, mean, var);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}
