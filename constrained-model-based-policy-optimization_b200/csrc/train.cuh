// Shared by the two implementations of the ensemble training step: train.cu (fp32 / TF32 library GEMMs) and
// train_tc.cu (bf16 tcgen05 GEMMs with fused prologues and epilogues).
#pragma once
#include <algorithm>

#include "common.cuh"

// activation and its derivative in the IEEE expf / tanhf forms (not the MUFU approximations of the rollout)
__device__ __forceinline__ float train_sigmoidf(float x) { return 1.0f / (1.0f + expf(-x)); }

__device__ __forceinline__ float act_fwd(int act, float x) {
    switch (act) {
        case CMBPO_ACT_SWISH: return x * train_sigmoidf(x);          // fc.py:19
        case CMBPO_ACT_TANH: return tanhf(x);
        case CMBPO_ACT_RELU: return fmaxf(x, 0.f);
        case CMBPO_ACT_SIGMOID: return train_sigmoidf(x);
        default: return x;
    }
}

__device__ __forceinline__ float act_bwd(int act, float x) {
    switch (act) {
        case CMBPO_ACT_SWISH: { const float s = train_sigmoidf(x); return s * (1.0f + x * (1.0f - s)); }
        case CMBPO_ACT_TANH: { const float t = tanhf(x); return 1.0f - t * t; }
        case CMBPO_ACT_RELU: return x > 0.f ? 1.0f : 0.f;
        case CMBPO_ACT_SIGMOID: { const float s = train_sigmoidf(x); return s * (1.0f - s); }
        default: return 1.0f;
    }
}

__device__ __forceinline__ double block_sum_d(double v, double* sh) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) sh[w] = v;
    __syncthreads();
    double s = 0;
    if (threadIdx.x < 32) {
        s = (threadIdx.x < (blockDim.x >> 5)) ? sh[threadIdx.x] : 0.0;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
    }
    return s;       // valid in thread 0
}

// ---- bf16 training step (train_tc.cu) ------------------------------------------------------------------------
// Every bf16 tensor is a "panel image": the feature columns cut into 64-wide panels (zero-padded), each panel
// `rows` rows of 128 B in the 128-byte-swizzled layout of tc::panel_off, panels of one member back to back.
// Activations and gradients have rows = the batch rounded up to 128; W16 of layer l has rows = its input width
// rounded up to 64.
namespace train_tc {
inline int64_t rows_pad(int64_t bs) { return (bs + 127) / 128 * 128; }
__host__ __device__ inline int panels(int width) { return (width + 63) / 64; }
inline size_t act_bytes(int E, int64_t bs, int width) { return (size_t)E * rows_pad(bs) * panels(width) * 128; }
inline size_t w16_bytes(int E, int K, int H) { return (size_t)E * ((K + 63) / 64 * 64) * panels(H) * 128; }
inline int row_tiles(int64_t bs) { return (int)(rows_pad(bs) / 128); }
constexpr int MAX_LOSS_BLOCKS = 64;
// blocks per member of loss pass 1 (the grid of loss_pass1_kernel in train.cu)
inline int loss_blocks(int64_t bs, int D) { return (int)std::min<int64_t>((bs * D + 255) / 256, MAX_LOSS_BLOCKS); }

struct Adam { float lr_t, b1, b2, eps, wd; };

// W [E, K, H] fp32 -> W16 panel image
int pack_w16(cmbpo_ctx* ctx, const float* W, int E, int K, int H, uint8_t* w16);
// x [E, bs, in] -> scaled input panel image (mu == NULL: no input scaler)
int scale_in(cmbpo_ctx* ctx, const float* x, const float* mu, const float* sig, int E, int64_t bs, int in, uint8_t* xs);
// the two loss passes on the raw outputs z [E, bs, W]: pass 1 writes per-block sums to lpart
// [E, loss_blocks, 3]; pass 2 adds them in order and writes loss[E], the output gradient G_L as a panel image and
// its per-row-tile column sums part [E, row_tiles, W]
int loss_grad(cmbpo_ctx* ctx, const float* z, const float* y, const float* mu_out, const float* sig_out, int64_t bs,
              int D, int W, int prob, int E, double* lpart, float* loss, uint8_t* g, float* part);
// z [E, bs, H] = a . W16 + b (fp32); hidden layers also h = act(z) as a panel image
int forward(cmbpo_ctx* ctx, int E, int64_t bs, int K, int H, const uint8_t* a, const uint8_t* w16, const float* b,
            int act, float* z, uint8_t* h);
// G_{l-1} = (G_l . W16_l^T) * act'(z_{l-1}) as a panel image of width K, plus its column sums per row tile
int data_grad(cmbpo_ctx* ctx, int E, int64_t bs, int K, int H, const uint8_t* g, const uint8_t* w16,
              const float* z_prev, int act_prev, uint8_t* g_prev, float* part_prev);
// dW = a^T . G_l (stored in gW), Adam on W / m / v, new W16; db from the column sums, Adam on b
int weight_grad_adam(cmbpo_ctx* ctx, int E, int64_t bs, int K, int H, const uint8_t* a, const uint8_t* g,
                     const float* part, float* W, float* mW, float* vW, float* gW, float* b, float* mb, float* vb,
                     float* gb, uint8_t* w16, Adam opt);
}  // namespace train_tc
