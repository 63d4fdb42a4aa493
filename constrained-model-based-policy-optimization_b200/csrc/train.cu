// SURVEY.md section 8f-4: one gradient step of the ensemble (the body of the batch loop of PE.train,
// models/pens/pe.py:547-567): forward of every member on ITS OWN batch [E, bs, in] (fc.py:74-95, 3-D branch),
// the MSPE loss of pe.py:921-973 (or the MSE loss of pe.py:840-919 with inc_var_loss=False for the
// non-probabilistic value ensembles), weight decay (fc.py:168-169: wd_l * tf.nn.l2_loss(W_l)), back-propagation
// and tf.train.AdamOptimizer's update.
//
// The dense contractions (forward, dW = A^T dZ, dA = dZ W^T; batched over the E members) are plain library GEMMs:
// cublasSgemmStridedBatched, on the tensor cores when `math` = 1 (TF32).  Everything around them is fused into
// a few element-wise kernels of our own: input scaling, bias + activation (keeping the pre-activations), the loss
// and its output gradient (two passes: the loss couples all members through one scalar ratio), activation
// backward, bias gradients (column sums), decay + Adam.  `math` = 2 (bf16) runs the same step on the tcgen05
// GEMMs of train_tc.cu, which fuse that element-wise work into their prologues and epilogues (step_bf16 below).
#include <cublas_v2.h>

#include "train.cuh"

namespace {

constexpr int ML = CMBPO_MAX_LAYERS;

struct TrainState {
    float *mW[ML] = {}, *vW[ML] = {}, *mb[ML] = {}, *vb[ML] = {};   // Adam moments
    float *gW[ML] = {}, *gb[ML] = {};                               // gradients of the last step (without decay)
    int64_t step = 0;
    int64_t cap_bs = 0;
    float* xs = nullptr;                  // scaled inputs [E, bs, in]
    float *z[ML] = {}, *h[ML] = {};       // pre-activations (bias included) / activations per layer
    float *da = nullptr, *db_ = nullptr;  // gradient ping-pong buffers [E, bs, max width]
    double* sums = nullptr;               // [E][3] loss sums + scratch
    float* loss = nullptr;                // [E]
    cublasHandle_t blas = nullptr;
    // bf16 step (train_tc.cu): panel images of the operands, sized for cap_bs16 rows
    uint8_t* w16[ML] = {};                // bf16 copy of W_l
    bool w16_fresh = false;               // w16 equals the master weights rounded (only bf16 steps keep it so)
    int64_t cap_bs16 = 0;
    uint8_t* xs16 = nullptr;              // scaled inputs
    uint8_t* h16[ML] = {};                // hidden activations
    uint8_t* g16[2] = {};                 // pre-activation gradients, ping-pong
    float* part[2] = {};                  // per-row-tile column sums of g16 [E, row tiles, width], ping-pong
    float* z16[ML] = {};                  // fp32 pre-activations [E, bs, width] (the fp32 path's z is not shared)
    double* lpart = nullptr;              // loss pass 1's per-block sums [E, loss blocks, 3]
};

#define BLAS_TRY(expr)                                                                     \
    do {                                                                                   \
        cublasStatus_t st_ = (expr);                                                       \
        if (st_ != CUBLAS_STATUS_SUCCESS) { cmbpo_set_error("cuBLAS error %d at %s:%d", (int)st_, __FILE__, __LINE__); return 1; } \
    } while (0)

// pens/utils.py:156 on [E, bs, in]
__global__ void scale_in_kernel(const float* __restrict__ x, const float* __restrict__ mu, const float* __restrict__ sig,
                                int in, int64_t total, float* __restrict__ xs) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % in);
        xs[i] = mu ? __fdiv_rn(__fsub_rn(x[i], mu[c]), sig[c]) : x[i];
    }
}

// z <- z + b (kept for the backward pass); h <- act(z)
__global__ void bias_act_kernel(float* __restrict__ z, const float* __restrict__ b, int act, float* __restrict__ h,
                                int64_t bs, int H, int64_t total) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % H);
        const int64_t e = i / (bs * H);
        const float v = z[i] + b[e * H + c];
        z[i] = v;
        if (h) h[i] = act_fwd(act, v);
    }
}

// Loss pass 1, grid.y = member.  MSPE (pe.py:945-971): s = (mean - y~)^2, q = (exp(logvar) - s)^2, logvar^2;
// MSE (pe.py:914): s only.  y~ = scaler_out.transform(y) (pe.py:943).  sums[e] = {sum s, sum q, sum logvar^2}.
__global__ void loss_pass1_kernel(const float* __restrict__ out, const float* __restrict__ y, const float* __restrict__ mu_out,
                                  const float* __restrict__ sig_out, int64_t bs, int D, int W, int prob,
                                  double* __restrict__ sums) {
    __shared__ double sh[32];
    const int e = blockIdx.y;
    const int64_t n = bs * D;
    double a = 0, b = 0, c = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / D; const int d = (int)(i - r * D);
        const float* o = out + ((int64_t)e * bs + r) * W;
        float yt = y[((int64_t)e * bs + r) * D + d];
        if (mu_out) yt = __fdiv_rn(__fsub_rn(yt, mu_out[d]), sig_out[d]);
        const float df = o[d] - yt, s = df * df;
        a += (double)s;
        if (prob) {
            const float lv = o[D + d], v = expf(lv), t = v - s;
            b += (double)(t * t);
            c += (double)(lv * lv);
        }
    }
    a = block_sum_d(a, sh); b = block_sum_d(b, sh); c = block_sum_d(c, sh);
    if (threadIdx.x == 0) { atomicAdd(sums + e * 3 + 0, a); atomicAdd(sums + e * 3 + 1, b); atomicAdd(sums + e * 3 + 2, c); }
}

// Loss pass 2: per-member loss value and the gradient with respect to the raw outputs.
//   MSPE: total_e = mean s + ratio * mean q + 0.05 * mean_all logvar^2, ratio = 0.05 * mean_all s / mean_all q with
//         stop-gradients on s inside q and on the ratio (pe.py:961-971); train_loss = sum_e total_e, so the scalar
//         regulariser counts E times:  d/dmean = 2 (mean - y~) / n,  d/dlogvar = (2 ratio (v - s) v + 0.1 logvar) / n.
//   MSE:  total_e = mean 0.5 s  ->  d/dmean = (mean - y~) / n.                      (n = bs * D per member)
__global__ void loss_pass2_kernel(const float* __restrict__ out, const float* __restrict__ y, const float* __restrict__ mu_out,
                                  const float* __restrict__ sig_out, int64_t bs, int D, int W, int prob, int E,
                                  const double* __restrict__ sums, float* __restrict__ dout, float* __restrict__ loss) {
    const int e = blockIdx.y;
    const int64_t n = bs * D;
    double ts = 0, tq = 0, tl = 0;
    for (int k = 0; k < E; ++k) { ts += sums[k * 3]; tq += sums[k * 3 + 1]; tl += sums[k * 3 + 2]; }
    const float ratio = prob ? (float)(0.05 * ts / tq) : 0.f;
    const float inv_n = 1.0f / (float)n;
    if (loss && blockIdx.x == 0 && threadIdx.x == 0) {
        if (prob) loss[e] = (float)(sums[e * 3] / (double)n + (double)ratio * sums[e * 3 + 1] / (double)n + 0.05 * tl / ((double)n * E));
        else loss[e] = (float)(0.5 * sums[e * 3] / (double)n);
    }
    if (!dout) return;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / D; const int d = (int)(i - r * D);
        const int64_t row = ((int64_t)e * bs + r) * W;
        float yt = y[((int64_t)e * bs + r) * D + d];
        if (mu_out) yt = __fdiv_rn(__fsub_rn(yt, mu_out[d]), sig_out[d]);
        const float df = out[row + d] - yt;
        if (prob) {
            const float s = df * df, lv = out[row + D + d], v = expf(lv);
            dout[row + d] = 2.0f * df * inv_n;
            dout[row + D + d] = (2.0f * ratio * (v - s) * v + 0.1f * lv) * inv_n;
        } else {
            dout[row + d] = df * inv_n;
        }
    }
}

// dz <- dh * act'(z)   (in place on the gradient buffer)
__global__ void act_bwd_kernel(float* __restrict__ g, const float* __restrict__ z, int act, int64_t total) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x)
        g[i] *= act_bwd(act, z[i]);
}

// db[e, c] = sum_r dz[e, r, c]: block = 32 columns x 8 row lanes, grid (ceil(H/32), E)
__global__ void bias_grad_kernel(const float* __restrict__ dz, int64_t bs, int H, float* __restrict__ db) {
    __shared__ float sh[8][33];
    const int c = blockIdx.x * 32 + threadIdx.x, e = blockIdx.y;
    float s = 0.f;
    if (c < H)
        for (int64_t r = threadIdx.y; r < bs; r += 8) s += dz[((int64_t)e * bs + r) * H + c];
    sh[threadIdx.y][threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.y == 0 && c < H) {
        float t = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) t += sh[k][threadIdx.x];
        db[(int64_t)e * H + c] = t;
    }
}

// g = grad + wd * w;  m, v, w updated as tf.train.AdamOptimizer does (lr_t carries the bias corrections)
__global__ void adam_kernel(float* __restrict__ w, const float* __restrict__ grad, float* __restrict__ m, float* __restrict__ v,
                            int64_t n, float wd, float lr_t, float b1, float b2, float eps) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float g = grad[i] + wd * w[i];
        const float mi = b1 * m[i] + (1.0f - b1) * g;
        const float vi = b2 * v[i] + (1.0f - b2) * g * g;
        m[i] = mi; v[i] = vi;
        w[i] -= lr_t * mi / (sqrtf(vi) + eps);
    }
}

int grid_of(cmbpo_ctx* ctx, int64_t n) { return (int)std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * 16); }

TrainState* state_of(cmbpo_ctx* ctx, int which) { return reinterpret_cast<TrainState*>(ctx->train[which]); }

int ensure_buffers(cmbpo_ctx* ctx, Net& n, TrainState* st, int64_t bs) {
    if (bs <= st->cap_bs) return 0;
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    auto re = [&](float** p, size_t count) -> int {
        if (*p) cudaFree(*p);
        *p = nullptr;
        CUDA_TRY(cudaMalloc(p, count * sizeof(float)));
        return 0;
    };
    int maxw = n.dims[0];
    for (int l = 0; l < n.n_layers; ++l) maxw = std::max(maxw, n.dims[l + 1]);
    if (re(&st->xs, (size_t)n.E * bs * n.dims[0])) return 1;
    for (int l = 0; l < n.n_layers; ++l) {
        if (re(&st->z[l], (size_t)n.E * bs * n.dims[l + 1])) return 1;
        if (l + 1 < n.n_layers && re(&st->h[l], (size_t)n.E * bs * n.dims[l + 1])) return 1;
    }
    if (re(&st->da, (size_t)n.E * bs * maxw)) return 1;
    if (re(&st->db_, (size_t)n.E * bs * maxw)) return 1;
    st->cap_bs = bs;
    return 0;
}

int ensure_buffers_bf16(cmbpo_ctx* ctx, Net& n, TrainState* st, int64_t bs) {
    using namespace train_tc;
    if (!st->w16[0]) {
        for (int l = 0; l < n.n_layers; ++l) CUDA_TRY(cudaMalloc(&st->w16[l], w16_bytes(n.E, n.dims[l], n.dims[l + 1])));
        CUDA_TRY(cudaMalloc(&st->lpart, (size_t)n.E * MAX_LOSS_BLOCKS * 3 * sizeof(double)));
        st->w16_fresh = false;
    }
    if (rows_pad(bs) <= st->cap_bs16) return 0;
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    auto re = [&](void** p, size_t bytes) -> int {
        if (*p) cudaFree(*p);
        *p = nullptr;
        CUDA_TRY(cudaMalloc(p, bytes));
        return 0;
    };
    int maxw = 0;
    for (int l = 0; l < n.n_layers; ++l) maxw = std::max(maxw, n.dims[l + 1]);
    if (re((void**)&st->xs16, act_bytes(n.E, bs, n.dims[0]))) return 1;
    for (int l = 0; l < n.n_layers; ++l) {
        if (l + 1 < n.n_layers && re((void**)&st->h16[l], act_bytes(n.E, bs, n.dims[l + 1]))) return 1;
        if (re((void**)&st->z16[l], (size_t)n.E * rows_pad(bs) * n.dims[l + 1] * sizeof(float))) return 1;
    }
    for (int i = 0; i < 2; ++i) {
        if (re((void**)&st->g16[i], act_bytes(n.E, bs, maxw))) return 1;
        if (re((void**)&st->part[i], (size_t)n.E * row_tiles(bs) * maxw * sizeof(float))) return 1;
    }
    st->cap_bs16 = rows_pad(bs);
    return 0;
}

// C[e] (m x n, row-major) = op(A[e]) op(B[e]); row-major operands handed to column-major cuBLAS as transposes
int gemm_nn(TrainState* st, int E, int m, int n, int k, const float* A, const float* B, float* C) {       // C = A[m,k] B[k,n]
    const float one = 1.f, zero = 0.f;
    BLAS_TRY(cublasSgemmStridedBatched(st->blas, CUBLAS_OP_N, CUBLAS_OP_N, n, m, k, &one, B, n, (long long)k * n, A, k,
                                       (long long)m * k, &zero, C, n, (long long)m * n, E));
    return 0;
}
int gemm_tn(TrainState* st, int E, int m, int n, int k, const float* A, const float* B, float* C) {       // C[m,n] = A[k,m]^T B[k,n]
    const float one = 1.f, zero = 0.f;
    BLAS_TRY(cublasSgemmStridedBatched(st->blas, CUBLAS_OP_N, CUBLAS_OP_T, n, m, k, &one, B, n, (long long)k * n, A, m,
                                       (long long)k * m, &zero, C, n, (long long)m * n, E));
    return 0;
}
int gemm_nt(TrainState* st, int E, int m, int n, int k, const float* A, const float* B, float* C) {       // C[m,n] = A[m,k] B[n,k]^T
    const float one = 1.f, zero = 0.f;
    BLAS_TRY(cublasSgemmStridedBatched(st->blas, CUBLAS_OP_T, CUBLAS_OP_N, n, m, k, &one, B, k, (long long)n * k, A, k,
                                       (long long)m * k, &zero, C, n, (long long)m * n, E));
    return 0;
}

// forward of all members on their own batches; leaves z / h in the state; raw outputs = z[last]
int forward(cmbpo_ctx* ctx, Net& n, TrainState* st, const float* x, int64_t bs) {
    const int64_t tot_in = (int64_t)n.E * bs * n.dims[0];
    scale_in_kernel<<<grid_of(ctx, tot_in), 256, 0, ctx->stream>>>(x, n.has_in ? n.mu_in : nullptr, n.sig_in, n.dims[0], tot_in, st->xs);
    ctx->launches++;
    const float* a = st->xs;
    for (int l = 0; l < n.n_layers; ++l) {
        const int K = n.dims[l], H = n.dims[l + 1];
        if (gemm_nn(st, n.E, (int)bs, H, K, a, n.W[l], st->z[l])) return 1;
        const int64_t tot = (int64_t)n.E * bs * H;
        const bool hidden = l + 1 < n.n_layers;
        bias_act_kernel<<<grid_of(ctx, tot), 256, 0, ctx->stream>>>(st->z[l], n.b[l], n.acts[l], hidden ? st->h[l] : nullptr, bs, H, tot);
        ctx->launches++;
        a = st->h[l];
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int check_net(cmbpo_ctx* ctx, int which, int64_t bs) {
    CMBPO_CHECK(ctx && which >= 0 && which < CMBPO_NET_COUNT, "bad arguments");
    Net& n = ctx->nets[which];
    CMBPO_CHECK(n.loaded, "network %d not loaded", which);
    CMBPO_CHECK(state_of(ctx, which), "call cmbpo_ens_train_begin first");
    CMBPO_CHECK(bs > 0 && bs < (1 << 24), "bad batch size");
    CMBPO_CHECK(n.acts[n.n_layers - 1] == CMBPO_ACT_NONE, "training expects a linear output layer");
    return 0;
}

// the bf16 step (train_tc.cu header): 3L + 2 launches, L more when W16 has to be rebuilt first
int step_bf16(cmbpo_ctx* ctx, Net& n, TrainState* st, const float* x, const float* y, int64_t bs,
              const cmbpo_train_cfg* cfg, float* loss_out) {
    if (ensure_buffers_bf16(ctx, n, st, bs)) return 1;
    const int L = n.n_layers, W = n.dims[L], prob = n.probabilistic ? 1 : 0;
    if (!st->w16_fresh) {
        for (int l = 0; l < L; ++l)
            if (train_tc::pack_w16(ctx, n.W[l], n.E, n.dims[l], n.dims[l + 1], st->w16[l])) return 1;
        st->w16_fresh = true;
    }
    if (train_tc::scale_in(ctx, x, n.has_in ? n.mu_in : nullptr, n.sig_in, n.E, bs, n.dims[0], st->xs16)) return 1;
    for (int l = 0; l < L; ++l) {
        const uint8_t* a = l == 0 ? st->xs16 : st->h16[l - 1];
        if (train_tc::forward(ctx, n.E, bs, n.dims[l], n.dims[l + 1], a, st->w16[l], n.b[l], n.acts[l], st->z16[l],
                              l + 1 < L ? st->h16[l] : nullptr)) return 1;
    }
    const float* mu_o = n.has_out ? n.mu_out : nullptr;
    int gi = 0;
    if (train_tc::loss_grad(ctx, st->z16[L - 1], y, mu_o, n.sig_out, bs, n.D, W, prob, n.E, st->lpart,
                            loss_out ? loss_out : st->loss, st->g16[gi], st->part[gi])) return 1;
    st->step += 1;
    const double t = (double)st->step;
    const float lr_t = (float)((double)cfg->lr * sqrt(1.0 - pow((double)cfg->beta2, t)) / (1.0 - pow((double)cfg->beta1, t)));
    for (int l = L - 1; l >= 0; --l) {
        const int K = n.dims[l], H = n.dims[l + 1];
        if (l > 0 && train_tc::data_grad(ctx, n.E, bs, K, H, st->g16[gi], st->w16[l], st->z16[l - 1], n.acts[l - 1],
                                         st->g16[gi ^ 1], st->part[gi ^ 1])) return 1;
        const train_tc::Adam opt = {lr_t, cfg->beta1, cfg->beta2, cfg->eps, cfg->weight_decay[l]};
        if (train_tc::weight_grad_adam(ctx, n.E, bs, K, H, l == 0 ? st->xs16 : st->h16[l - 1], st->g16[gi], st->part[gi],
                                       n.W[l], st->mW[l], st->vW[l], st->gW[l], n.b[l], st->mb[l], st->vb[l], st->gb[l],
                                       st->w16[l], opt)) return 1;
        gi ^= 1;
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

}  // namespace

void train_free(cmbpo_ctx* ctx, int which) {
    TrainState* st = state_of(ctx, which);
    if (!st) return;
    for (int l = 0; l < ML; ++l) {
        float* p[] = {st->mW[l], st->vW[l], st->mb[l], st->vb[l], st->gW[l], st->gb[l], st->z[l], st->h[l]};
        for (float* q : p) if (q) cudaFree(q);
        if (st->w16[l]) cudaFree(st->w16[l]);
        if (st->h16[l]) cudaFree(st->h16[l]);
        if (st->z16[l]) cudaFree(st->z16[l]);
    }
    float* p[] = {st->xs, st->da, st->db_, st->loss, st->part[0], st->part[1]};
    for (float* q : p) if (q) cudaFree(q);
    uint8_t* p16[] = {st->xs16, st->g16[0], st->g16[1]};
    for (uint8_t* q : p16) if (q) cudaFree(q);
    if (st->sums) cudaFree(st->sums);
    if (st->lpart) cudaFree(st->lpart);
    if (st->blas) cublasDestroy(st->blas);
    delete st;
    ctx->train[which] = nullptr;
}

extern "C" int cmbpo_ens_train_begin(cmbpo_ctx* ctx, int which) {
    CMBPO_CHECK(ctx && which >= 0 && which < CMBPO_NET_COUNT, "bad arguments");
    Net& n = ctx->nets[which];
    CMBPO_CHECK(n.loaded, "network %d not loaded", which);
    if (state_of(ctx, which)) return 0;              // optimiser state persists across train() calls, like TF's
    CUDA_TRY(cudaSetDevice(ctx->device));
    TrainState* st = new TrainState();
    ctx->train[which] = st;
    for (int l = 0; l < n.n_layers; ++l) {
        const size_t nw = (size_t)n.E * n.dims[l] * n.dims[l + 1], nb = (size_t)n.E * n.dims[l + 1];
        float** wp[] = {&st->mW[l], &st->vW[l], &st->gW[l]};
        float** bp[] = {&st->mb[l], &st->vb[l], &st->gb[l]};
        for (float** q : wp) { CUDA_TRY(cudaMalloc(q, nw * sizeof(float))); CUDA_TRY(cudaMemsetAsync(*q, 0, nw * sizeof(float), ctx->stream)); }
        for (float** q : bp) { CUDA_TRY(cudaMalloc(q, nb * sizeof(float))); CUDA_TRY(cudaMemsetAsync(*q, 0, nb * sizeof(float), ctx->stream)); }
    }
    CUDA_TRY(cudaMalloc(&st->sums, (size_t)CMBPO_MAX_E * 3 * sizeof(double)));
    CUDA_TRY(cudaMalloc(&st->loss, CMBPO_MAX_E * sizeof(float)));
    BLAS_TRY(cublasCreate(&st->blas));
    return 0;
}

extern "C" int cmbpo_ens_train_loss(cmbpo_ctx* ctx, int which, const float* x, const float* y, int64_t bs, float* loss_out) {
    if (check_net(ctx, which, bs)) return 1;
    CMBPO_CHECK(x && y && loss_out, "null argument");
    Net& n = ctx->nets[which];
    TrainState* st = state_of(ctx, which);
    CMBPO_CHECK(n.E <= CMBPO_MAX_E, "too many members");
    if (ensure_buffers(ctx, n, st, bs)) return 1;
    BLAS_TRY(cublasSetStream(st->blas, ctx->stream));
    BLAS_TRY(cublasSetMathMode(st->blas, CUBLAS_DEFAULT_MATH));
    if (forward(ctx, n, st, x, bs)) return 1;
    const int W = n.dims[n.n_layers];
    CUDA_TRY(cudaMemsetAsync(st->sums, 0, (size_t)n.E * 3 * sizeof(double), ctx->stream));
    dim3 grid((unsigned)std::min<int64_t>((bs * n.D + 255) / 256, 64), n.E);
    // `self.loss` (pe.py:264, 271): _nll_loss with inc_var_loss=False = mean 0.5 (mean - y~)^2 for every loss type
    loss_pass1_kernel<<<grid, 256, 0, ctx->stream>>>(st->z[n.n_layers - 1], y, n.has_out ? n.mu_out : nullptr, n.sig_out, bs, n.D, W, 0, st->sums);
    loss_pass2_kernel<<<dim3(1, n.E), 32, 0, ctx->stream>>>(st->z[n.n_layers - 1], y, nullptr, nullptr, bs, n.D, W, 0, n.E, st->sums, nullptr, loss_out);
    ctx->launches += 2;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int cmbpo_ens_train_step(cmbpo_ctx* ctx, int which, const float* x, const float* y, int64_t bs,
                                    const cmbpo_train_cfg* cfg, float* loss_out) {
    if (check_net(ctx, which, bs)) return 1;
    CMBPO_CHECK(x && y && cfg, "null argument");
    Net& n = ctx->nets[which];
    TrainState* st = state_of(ctx, which);
    CMBPO_CHECK(n.E <= CMBPO_MAX_E, "too many members");
    const int prob = n.probabilistic ? 1 : 0;
    CMBPO_CHECK((cfg->loss == CMBPO_LOSS_MSPE && prob) || (cfg->loss == CMBPO_LOSS_MSE && !prob),
                "loss %d does not fit this network (MSPE: probabilistic, MSE: not)", cfg->loss);
    CMBPO_CHECK(cfg->math == CMBPO_TRAIN_FP32 || cfg->math == CMBPO_TRAIN_TF32 || cfg->math == CMBPO_TRAIN_BF16,
                "math %d is not one of 0 (fp32), 1 (TF32), 2 (bf16)", cfg->math);
    if (cfg->math == CMBPO_TRAIN_BF16) return step_bf16(ctx, n, st, x, y, bs, cfg, loss_out);
    st->w16_fresh = false;                           // this step moves the master weights away from W16
    if (ensure_buffers(ctx, n, st, bs)) return 1;
    BLAS_TRY(cublasSetStream(st->blas, ctx->stream));
    BLAS_TRY(cublasSetMathMode(st->blas, cfg->math ? CUBLAS_TF32_TENSOR_OP_MATH : CUBLAS_DEFAULT_MATH));
    if (forward(ctx, n, st, x, bs)) return 1;
    const int L = n.n_layers, W = n.dims[L];
    // loss and d loss / d raw outputs
    CUDA_TRY(cudaMemsetAsync(st->sums, 0, (size_t)n.E * 3 * sizeof(double), ctx->stream));
    dim3 grid((unsigned)std::min<int64_t>((bs * n.D + 255) / 256, 64), n.E);
    const float* mu_o = n.has_out ? n.mu_out : nullptr;
    loss_pass1_kernel<<<grid, 256, 0, ctx->stream>>>(st->z[L - 1], y, mu_o, n.sig_out, bs, n.D, W, prob, st->sums);
    float* g = st->da;          // gradient with respect to the current layer's pre-activation
    float* g2 = st->db_;
    if (prob) CUDA_TRY(cudaMemsetAsync(g, 0, (size_t)n.E * bs * W * sizeof(float), ctx->stream));
    loss_pass2_kernel<<<grid, 256, 0, ctx->stream>>>(st->z[L - 1], y, mu_o, n.sig_out, bs, n.D, W, prob, n.E, st->sums, g,
                                                    loss_out ? loss_out : st->loss);
    ctx->launches += 2;
    for (int l = L - 1; l >= 0; --l) {
        const int K = n.dims[l], H = n.dims[l + 1];
        const float* a = (l == 0) ? st->xs : st->h[l - 1];
        if (gemm_tn(st, n.E, K, H, (int)bs, a, g, st->gW[l])) return 1;                 // dW = A^T dZ
        bias_grad_kernel<<<dim3((H + 31) / 32, n.E), dim3(32, 8), 0, ctx->stream>>>(g, bs, H, st->gb[l]);
        ctx->launches++;
        if (l > 0) {
            if (gemm_nt(st, n.E, (int)bs, K, H, g, n.W[l], g2)) return 1;               // dA = dZ W^T
            const int64_t tot = (int64_t)n.E * bs * K;
            act_bwd_kernel<<<grid_of(ctx, tot), 256, 0, ctx->stream>>>(g2, st->z[l - 1], n.acts[l - 1], tot);
            ctx->launches++;
            std::swap(g, g2);
        }
    }
    // decay + Adam (tf.train.AdamOptimizer: lr_t = lr sqrt(1 - b2^t) / (1 - b1^t))
    st->step += 1;
    const double t = (double)st->step;
    const float lr_t = (float)((double)cfg->lr * sqrt(1.0 - pow((double)cfg->beta2, t)) / (1.0 - pow((double)cfg->beta1, t)));
    for (int l = 0; l < L; ++l) {
        const int64_t nw = (int64_t)n.E * n.dims[l] * n.dims[l + 1], nb = (int64_t)n.E * n.dims[l + 1];
        adam_kernel<<<grid_of(ctx, nw), 256, 0, ctx->stream>>>(n.W[l], st->gW[l], st->mW[l], st->vW[l], nw, cfg->weight_decay[l], lr_t,
                                                              cfg->beta1, cfg->beta2, cfg->eps);
        adam_kernel<<<grid_of(ctx, nb), 256, 0, ctx->stream>>>(n.b[l], st->gb[l], st->mb[l], st->vb[l], nb, 0.f, lr_t, cfg->beta1,
                                                              cfg->beta2, cfg->eps);
        ctx->launches += 2;
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int cmbpo_ens_train_grads(cmbpo_ctx* ctx, int which, int layer, float* dW, float* db) {
    CMBPO_CHECK(ctx && which >= 0 && which < CMBPO_NET_COUNT && state_of(ctx, which), "no training state");
    Net& n = ctx->nets[which];
    CMBPO_CHECK(layer >= 0 && layer < n.n_layers, "bad layer");
    TrainState* st = state_of(ctx, which);
    if (dW) CUDA_TRY(cudaMemcpyAsync(dW, st->gW[layer], (size_t)n.E * n.dims[layer] * n.dims[layer + 1] * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
    if (db) CUDA_TRY(cudaMemcpyAsync(db, st->gb[layer], (size_t)n.E * n.dims[layer + 1] * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
    return 0;
}

// checkpointing: one layer's Adam moments and the slot's step counter (the bias correction of lr_t depends on it)
extern "C" int cmbpo_ens_train_state_get(cmbpo_ctx* ctx, int which, int layer, float* mW, float* vW, float* mb, float* vb,
                                         int64_t* step_host) {
    CMBPO_CHECK(ctx && which >= 0 && which < CMBPO_NET_COUNT, "bad arguments");
    Net& n = ctx->nets[which];
    CMBPO_CHECK(n.loaded, "network %d not loaded", which);
    CMBPO_CHECK(layer >= 0 && layer < n.n_layers, "bad layer");
    TrainState* st = state_of(ctx, which);
    if (!st) {
        if (step_host) *step_host = -1;
        return 0;
    }
    const size_t nw = (size_t)n.E * n.dims[layer] * n.dims[layer + 1] * sizeof(float), nb = (size_t)n.E * n.dims[layer + 1] * sizeof(float);
    if (mW) CUDA_TRY(cudaMemcpyAsync(mW, st->mW[layer], nw, cudaMemcpyDeviceToDevice, ctx->stream));
    if (vW) CUDA_TRY(cudaMemcpyAsync(vW, st->vW[layer], nw, cudaMemcpyDeviceToDevice, ctx->stream));
    if (mb) CUDA_TRY(cudaMemcpyAsync(mb, st->mb[layer], nb, cudaMemcpyDeviceToDevice, ctx->stream));
    if (vb) CUDA_TRY(cudaMemcpyAsync(vb, st->vb[layer], nb, cudaMemcpyDeviceToDevice, ctx->stream));
    if (step_host) *step_host = st->step;
    return 0;
}

extern "C" int cmbpo_ens_train_state_set(cmbpo_ctx* ctx, int which, int layer, const float* mW, const float* vW,
                                         const float* mb, const float* vb, int64_t step) {
    CMBPO_CHECK(ctx && which >= 0 && which < CMBPO_NET_COUNT, "bad arguments");
    Net& n = ctx->nets[which];
    CMBPO_CHECK(n.loaded, "network %d not loaded", which);
    CMBPO_CHECK(layer >= 0 && layer < n.n_layers, "bad layer");
    CMBPO_CHECK(step >= 0, "bad step count %lld", (long long)step);
    if (cmbpo_ens_train_begin(ctx, which)) return 1;
    TrainState* st = state_of(ctx, which);
    const size_t nw = (size_t)n.E * n.dims[layer] * n.dims[layer + 1] * sizeof(float), nb = (size_t)n.E * n.dims[layer + 1] * sizeof(float);
    if (mW) CUDA_TRY(cudaMemcpyAsync(st->mW[layer], mW, nw, cudaMemcpyDeviceToDevice, ctx->stream));
    if (vW) CUDA_TRY(cudaMemcpyAsync(st->vW[layer], vW, nw, cudaMemcpyDeviceToDevice, ctx->stream));
    if (mb) CUDA_TRY(cudaMemcpyAsync(st->mb[layer], mb, nb, cudaMemcpyDeviceToDevice, ctx->stream));
    if (vb) CUDA_TRY(cudaMemcpyAsync(st->vb[layer], vb, nb, cudaMemcpyDeviceToDevice, ctx->stream));
    st->step = step;
    st->w16_fresh = false;                           // the next bf16 step re-packs W16 from the master weights
    return 0;
}

extern "C" int cmbpo_net_get_weights(cmbpo_ctx* ctx, int which, int layer, float* W, float* b) {
    CMBPO_CHECK(ctx && which >= 0 && which < CMBPO_NET_COUNT, "bad arguments");
    Net& n = ctx->nets[which];
    CMBPO_CHECK(n.loaded && layer >= 0 && layer < n.n_layers, "bad layer");
    if (W) CUDA_TRY(cudaMemcpyAsync(W, n.W[layer], (size_t)n.E * n.dims[layer] * n.dims[layer + 1] * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
    if (b) CUDA_TRY(cudaMemcpyAsync(b, n.b[layer], (size_t)n.E * n.dims[layer + 1] * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
    return 0;
}

// after training: new scalers (optional), new elites (optional), re-pack the tcgen05 weight streams so that
// rollouts / predictions see the trained weights (pe.py:601-607: _end_train picks the elites)
extern "C" int cmbpo_ens_train_end(cmbpo_ctx* ctx, int which, const int* elite_inds, int n_elite) {
    CMBPO_CHECK(ctx && which >= 0 && which < CMBPO_NET_COUNT, "bad arguments");
    Net& n = ctx->nets[which];
    CMBPO_CHECK(n.loaded, "network %d not loaded", which);
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (elite_inds && n_elite > 0) {
        for (int i = 0; i < n_elite; ++i) CMBPO_CHECK(elite_inds[i] >= 0 && elite_inds[i] < n.E, "elite index out of range");
        if (n.elite) cudaFree(n.elite);
        CUDA_TRY(cudaMalloc(&n.elite, n_elite * sizeof(int)));
        CUDA_TRY(cudaMemcpy(n.elite, elite_inds, n_elite * sizeof(int), cudaMemcpyHostToDevice));
        n.n_elite = n_elite;
    }
    if (ens_tc_supported(n)) {
        for (int i = 0; i < 3; ++i) if (n.tc_pack[i]) { cudaFree(n.tc_pack[i]); n.tc_pack[i] = nullptr; }
        if (n.tc_bias) { cudaFree(n.tc_bias); n.tc_bias = nullptr; }
        if (ens_tc_prepare(ctx, n)) return 1;
    }
    if (which != CMBPO_NET_DYN && policy_pack_build(ctx)) return 1;
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// new scaler statistics for a loaded net (TensorStandardScaler.fit, pens/utils.py:119-138; the running merge is
// done by the caller): var -> sigma = max(sqrt(var), 1e-2), 2 log sigma
__global__ void prep_scaler2_kernel(const float* var, int n, float* sig, float* l2s) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float s = fmaxf(sqrtf(var[i]), 1e-2f);
    sig[i] = s;
    if (l2s) l2s[i] = __fmul_rn(2.0f, logf(s));
}

extern "C" int cmbpo_net_set_scalers(cmbpo_ctx* ctx, int which, const float* mu_in, const float* var_in,
                                     const float* mu_out, const float* var_out) {
    CMBPO_CHECK(ctx && which >= 0 && which < CMBPO_NET_COUNT, "bad arguments");
    Net& n = ctx->nets[which];
    CMBPO_CHECK(n.loaded, "network %d not loaded", which);
    CMBPO_CHECK((mu_in == nullptr) == (var_in == nullptr) && (mu_out == nullptr) == (var_out == nullptr),
                "scaler mean and variance must be given together");
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    float* tmp;
    CUDA_TRY(cudaMalloc(&tmp, (size_t)std::max(n.dims[0], n.D) * sizeof(float)));
    if (mu_in) {
        if (!n.mu_in) { CUDA_TRY(cudaMalloc(&n.mu_in, n.dims[0] * sizeof(float))); CUDA_TRY(cudaMalloc(&n.sig_in, n.dims[0] * sizeof(float))); }
        CUDA_TRY(cudaMemcpy(n.mu_in, mu_in, n.dims[0] * sizeof(float), cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(tmp, var_in, n.dims[0] * sizeof(float), cudaMemcpyHostToDevice));
        prep_scaler2_kernel<<<cdiv(n.dims[0], 128), 128, 0, ctx->stream>>>(tmp, n.dims[0], n.sig_in, nullptr);
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        n.has_in = true;
    }
    if (mu_out) {
        if (!n.mu_out) {
            CUDA_TRY(cudaMalloc(&n.mu_out, n.D * sizeof(float))); CUDA_TRY(cudaMalloc(&n.sig_out, n.D * sizeof(float)));
            CUDA_TRY(cudaMalloc(&n.l2s_out, n.D * sizeof(float)));
        }
        CUDA_TRY(cudaMemcpy(n.mu_out, mu_out, n.D * sizeof(float), cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(tmp, var_out, n.D * sizeof(float), cudaMemcpyHostToDevice));
        prep_scaler2_kernel<<<cdiv(n.D, 128), 128, 0, ctx->stream>>>(tmp, n.D, n.sig_out, n.l2s_out);
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        n.has_out = true;
    }
    cudaFree(tmp);
    CUDA_TRY(cudaGetLastError());
    // the merged policy pack copies V's input scaler and folds every member's scaler into its first layer
    if (which != CMBPO_NET_DYN && policy_pack_build(ctx)) return 1;
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}
