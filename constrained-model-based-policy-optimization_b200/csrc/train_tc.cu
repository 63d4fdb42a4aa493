// The bf16 ensemble training step (cmbpo_train_cfg.math = CMBPO_TRAIN_BF16): the same step as train.cu -- forward
// of every member on its own batch, MSPE / MSE loss, backward, weight decay and tf.train.AdamOptimizer's update --
// with its GEMMs on tcgen05 (kind::f16, bf16 operands, M = 128 rows per CTA, N = 64, fp32 accumulate in tensor
// memory) and the element-wise work fused into their prologues and epilogues.
//
// Numerics (tests/train_oracle_bf16.py with round_bf16=True mirrors them):
//   rounded to bf16 (round-to-nearest-even from the fp32 value): the scaled input xs, the weight copy W16, every
//     hidden activation h_l = act(z_l), every gradient G_l with respect to a pre-activation where it becomes a
//     GEMM operand;
//   fp32: accumulation, bias addition, the pre-activations z_l (kept for the backward pass), the raw outputs the
//     loss reads, the loss (the two passes of train.cu), the bias gradients (column sums of the fp32 gradient,
//     before it is rounded), dW, db, the master weights, Adam's moments and the decay;
//   activations: the IEEE expf / tanhf forms of train.cuh, so operand rounding is the only difference from fp32.
//   bf16, not fp16: the output gradient carries 1 / (bs D), about 1e-5 .. 1e-6 at bs = 256, below fp16's normal
//   range; bf16 has fp32's exponent range, so no loss scaling is needed.
//   Deterministic: the bias-gradient sums run in a fixed order (128 rows of a tile in order, then the tiles in
//   order), and loss pass 1 writes per-block partial sums that pass 2 adds in block order; no floating-point
//   atomics.
//
// One GEMM kernel, three uses (the same panel bytes are read K-major or MN-major; only the descriptors differ):
//   FWD   l: z_l = a_{l-1} [bs, K] . W16_l [K, H]       A K-major, B MN-major; + b, store z; hidden: h = act(z)
//   DGRAD l: G_{l-1} = G_l [bs, H] . W16_l^T            A K-major, B K-major;  * act'(z_{l-1}), column sums
//   WGRAD l: dW_l = a_{l-1}^T . G_l (sum over bs rows)  A MN-major, B MN-major; Adam on W_l, new W16_l; the CTAs
//            of the first M tile also reduce the db partial sums and update b_l.
// Launches per step: input scaling, L forwards, loss pass 1 (per-block partial sums), loss pass 2 (G_L + db
// partials), then
// from the last layer down DGRAD l (l > 0) and WGRAD l -- 3L + 2 (11 for 3 layers, 17 for 5).  A layer's W16 is
// rewritten by its WGRAD after its last reader (its DGRAD).  A step that finds W16 stale (a new optimiser state,
// or the step before was fp32 / TF32) first rebuilds it from the master weights: L more launches.
//
// Grid of a GEMM: (N tiles of 64, M tiles of 128, E).  A 512 x 512 layer at bs = 256 runs 8 x 2 x 7 = 112 CTAs.
// Warps 0-3 run the epilogue (warp w reads tensor-memory lanes 32w..32w+31, one accumulator row per thread),
// warp 4 copies 64-deep K chunks of both operands into a 3-stage ring (plain cp.async.bulk panel copies: every
// panel image is written by our own kernels), warp 5 allocates tensor memory and issues the MMAs.
#include "tc_common.cuh"
#include "train.cuh"

namespace {

using namespace tc;

constexpr int BM = 128, BN = 64, BK = 64;
constexpr int STAGES = 3;
constexpr uint32_t A_STAGE = BM * BK * 2, B_STAGE = BN * BK * 2;     // 16 KB, 8 KB
constexpr int SROW = BN + 1;                                          // fp32 staging row (conflict-free columns)
constexpr size_t SMEM_BYTES = 1024 + STAGES * (A_STAGE + B_STAGE) + (size_t)BM * SROW * 4 + BN * 4 + 64;
constexpr int WB = 16;                                                // WGRAD: elements whose loads issue together
constexpr int NTHREADS = 192;

enum { FWD = 0, DGRAD = 1, WGRAD = 2 };

struct GemmParams {
    int E, nk;
    int64_t bs, rpad;          // batch rows, padded to 128
    int K, H;                  // layer input / output width
    const uint8_t* a; int64_t a_member, a_panel; int a_npanels;
    const uint8_t* b; int64_t b_member, b_panel;
    // FWD
    const float* bias; int act; float* z; uint8_t* h;
    // DGRAD
    const float* z_prev; uint8_t* g_out; float* part_out;
    // WGRAD
    const float* part; float *W, *mW, *vW, *gW, *bb, *mb, *vb, *gb; uint8_t* w16; train_tc::Adam opt;
};

__device__ __forceinline__ void epi_sync() { asm volatile("bar.sync 1, 128;" ::: "memory"); }

// one 64-column row of a panel image as bf16 (8 swizzled 16-byte chunks)
__device__ __forceinline__ void store_panel_row(uint8_t* panel, int64_t r, const float (&v)[BN]) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        uint4 u;
        u.x = Cvt<1>::pack(v[8 * q + 0], v[8 * q + 1]);
        u.y = Cvt<1>::pack(v[8 * q + 2], v[8 * q + 3]);
        u.z = Cvt<1>::pack(v[8 * q + 4], v[8 * q + 5]);
        u.w = Cvt<1>::pack(v[8 * q + 6], v[8 * q + 7]);
        *reinterpret_cast<uint4*>(panel + (r >> 3) * 1024 + panel_off((int)(r & 7), q)) = u;
    }
}

// column sums of the staged [128][64] tile, rows in order (threads 0..63 of the epilogue, one column each)
__device__ __forceinline__ float column_sum(const float* stage, int j) {
    float s = 0.f;
#pragma unroll 8
    for (int r = 0; r < BM; ++r) s += stage[r * SROW + j];
    return s;
}

__device__ __forceinline__ void adam_elem(float& w, float& m, float& v, float grad, float wd, const train_tc::Adam& o) {
    const float g = grad + wd * w;                                    // as adam_kernel in train.cu
    const float mi = o.b1 * m + (1.0f - o.b1) * g;
    const float vi = o.b2 * v + (1.0f - o.b2) * g * g;
    m = mi; v = vi;
    w -= o.lr_t * mi / (sqrtf(vi) + o.eps);
}

template <int USE>
__global__ void __launch_bounds__(NTHREADS, 2) train_gemm_kernel(const GemmParams p) {
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment by an offset from smem_raw, not an integer round trip: the pointers below stay in the
    // shared state space, so staging accesses compile to LDS / STS and cannot alias the global operands
    uint8_t* sA = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* sB = sA + STAGES * A_STAGE;
    float* stage = reinterpret_cast<float*>(sB + STAGES * B_STAGE);
    float* sbias = stage + BM * SROW;                                  // FWD: this tile's 64 biases
    uint64_t* bar = reinterpret_cast<uint64_t*>(sbias + BN);           // FULL[S], EMPTY[S], ACC
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 2 * STAGES + 1);
    uint64_t* const FULL = bar;
    uint64_t* const EMPTY = bar + STAGES;
    uint64_t* const ACC = bar + 2 * STAGES;

    const int warp = threadIdx.x >> 5;
    const int nt = blockIdx.x, mt = blockIdx.y, e = blockIdx.z;
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(FULL + s, 1); mbar_init(EMPTY + s, 1); }
        mbar_init(ACC, 1);
        fence_barrier_init();
    }
    if (warp == 5) tmem_alloc(tmem_slot, 64);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    // A chunk: K-major = one 16 KB piece (128 rows of one panel); MN-major (WGRAD) = two 8 KB pieces (64 rows of
    // the two 64-column panels that hold M elements 0-63 / 64-127), the second absent past the last panel
    const int a_pieces = USE == WGRAD ? min(2, p.a_npanels - 2 * mt) : 1;
    if (warp == 4) {
        if (elect_one()) {
            const uint8_t* a0 = p.a + (int64_t)e * p.a_member;
            const uint8_t* b0 = p.b + (int64_t)e * p.b_member;
            for (int kc = 0; kc < p.nk; ++kc) {
                const int s = kc % STAGES;
                if (kc >= STAGES) mbar_wait(EMPTY + s, ((kc / STAGES) & 1) ^ 1);
                const uint32_t a_bytes = USE == WGRAD ? (uint32_t)a_pieces * (A_STAGE / 2) : A_STAGE;
                mbar_expect_tx(FULL + s, a_bytes + B_STAGE);
                if (USE == WGRAD) {
                    for (int j = 0; j < a_pieces; ++j)
                        bulk_g2s(sA + s * A_STAGE + j * (A_STAGE / 2), a0 + (2 * mt + j) * p.a_panel + (int64_t)kc * (BK * 128),
                                 A_STAGE / 2, FULL + s);
                } else {
                    bulk_g2s(sA + s * A_STAGE, a0 + kc * p.a_panel + (int64_t)mt * (BM * 128), A_STAGE, FULL + s);
                }
                // B: FWD / WGRAD read panel nt, K rows kc*64.. (MN-major); DGRAD reads panel kc, N rows nt*64.. (K-major)
                const uint8_t* bsrc = USE == DGRAD ? b0 + kc * p.b_panel + (int64_t)nt * (BN * 128)
                                                   : b0 + nt * p.b_panel + (int64_t)kc * (BK * 128);
                bulk_g2s(sB + s * B_STAGE, bsrc, B_STAGE, FULL + s);
            }
        }
    } else if (warp == 5) {
        if (elect_one()) {
            constexpr uint32_t idesc = idesc_f16_major(1, BN, USE == WGRAD, USE != DGRAD);
            // per K step of 16: +32 B inside a K-major row, +2 swizzle atoms (2048 B) down an MN-major panel
            constexpr uint64_t a_step = USE == WGRAD ? 2048 >> 4 : 32 >> 4;
            constexpr uint64_t b_step = USE == DGRAD ? 32 >> 4 : 2048 >> 4;
            for (int kc = 0; kc < p.nk; ++kc) {
                const int s = kc % STAGES;
                mbar_wait(FULL + s, (kc / STAGES) & 1);
                tc_fence_after();
                const uint32_t sa = smem_u32(sA + s * A_STAGE), sb = smem_u32(sB + s * B_STAGE);
                const uint64_t da = USE == WGRAD ? smem_desc_sw128_mn(sa, A_STAGE / 2) : smem_desc_sw128(sa);
                const uint64_t db = USE == DGRAD ? smem_desc_sw128(sb) : smem_desc_sw128_mn(sb, B_STAGE);
#pragma unroll
                for (int ks = 0; ks < BK / 16; ++ks) mma_f16(tmem, da + ks * a_step, db + ks * b_step, idesc, (kc | ks) != 0);
                mma_commit(EMPTY + s);
            }
            mma_commit(ACC);
        }
    } else {
        // ===== epilogue: thread i holds accumulator row i (64 fp32 columns) =====
        const int i = threadIdx.x;
        const int64_t n0 = (int64_t)nt * BN;
        // operands of the epilogue that do not depend on the accumulator load while the MMAs run
        if (USE == FWD && i < BN) sbias[i] = n0 + i < p.H ? __ldg(p.bias + (int64_t)e * p.H + n0 + i) : 0.f;
        if (USE == DGRAD) {                                        // z_{l-1} tile, coalesced
            const int K = p.K;
#pragma unroll 16
            for (int idx = i; idx < BM * BN; idx += BM) {
                const int rr = idx / BN, cc = idx % BN;
                const int64_t row = (int64_t)mt * BM + rr, col = n0 + cc;
                stage[rr * SROW + cc] = (row < p.bs && col < K) ? __ldg(p.z_prev + ((int64_t)e * p.bs + row) * K + col) : 0.f;
            }
        }
        epi_sync();
        float acc[BN];
        mbar_wait(ACC, 0);
        tc_fence_after();
        {
            uint32_t r[32];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + h * 32, r);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 32; ++j) acc[h * 32 + j] = __uint_as_float(r[j]);
            }
        }
        tc_fence_before();
        if (USE == FWD) {
            const int64_t r = (int64_t)mt * BM + i;
            const int H = p.H;
#pragma unroll
            for (int j = 0; j < BN; ++j) {
                const int64_t c = n0 + j;
                acc[j] = c < H ? acc[j] + sbias[j] : 0.f;
                stage[i * SROW + j] = acc[j];
            }
            if (p.h) {
                float hv[BN];
#pragma unroll
                for (int j = 0; j < BN; ++j) hv[j] = (r < p.bs && n0 + j < H) ? act_fwd(p.act, acc[j]) : 0.f;
                store_panel_row(p.h + (int64_t)e * p.rpad * train_tc::panels(H) * 128 + nt * p.rpad * 128, r, hv);
            }
            epi_sync();
            for (int idx = i; idx < BM * BN; idx += BM) {          // z, coalesced through the staging tile
                const int rr = idx / BN, cc = idx % BN;
                const int64_t row = (int64_t)mt * BM + rr, col = n0 + cc;
                if (row < p.bs && col < H) p.z[((int64_t)e * p.bs + row) * H + col] = stage[rr * SROW + cc];
            }
        } else if (USE == DGRAD) {
            const int K = p.K;
            const int64_t r = (int64_t)mt * BM + i;
#pragma unroll
            for (int j = 0; j < BN; ++j) {
                const float g = (r < p.bs && n0 + j < K) ? acc[j] * act_bwd(p.act, stage[i * SROW + j]) : 0.f;
                acc[j] = g;
                stage[i * SROW + j] = g;
            }
            store_panel_row(p.g_out + (int64_t)e * p.rpad * train_tc::panels(K) * 128 + nt * p.rpad * 128, r, acc);
            epi_sync();
            if (i < BN && n0 + i < K)
                p.part_out[((int64_t)e * gridDim.y + mt) * K + n0 + i] = column_sum(stage, i);
        } else {
            const int K = p.K, H = p.H;
#pragma unroll
            for (int j = 0; j < BN; ++j) stage[i * SROW + j] = acc[j];
            epi_sync();
            // dW, decay, Adam, coalesced over [K, H] rows; WB elements per thread at a time, all their loads
            // issued before any of their stores (a store to W / m / v may alias the next element's loads)
            for (int i0 = 0; i0 < BM * BN; i0 += WB * BM) {
                float w[WB], m[WB], v[WB];
                int64_t o[WB];
                bool ok[WB];
#pragma unroll
                for (int u = 0; u < WB; ++u) {
                    const int idx = i0 + u * BM + i, rr = idx / BN, cc = idx % BN;
                    const int64_t k = (int64_t)mt * BM + rr, col = n0 + cc;
                    ok[u] = k < K && col < H;
                    o[u] = ok[u] ? ((int64_t)e * K + k) * H + col : 0;
                    w[u] = ok[u] ? p.W[o[u]] : 0.f;
                    m[u] = ok[u] ? p.mW[o[u]] : 0.f;
                    v[u] = ok[u] ? p.vW[o[u]] : 0.f;
                }
#pragma unroll
                for (int u = 0; u < WB; ++u) {
                    if (!ok[u]) continue;
                    const int idx = i0 + u * BM + i, rr = idx / BN, cc = idx % BN;
                    const float dw = stage[rr * SROW + cc];
                    adam_elem(w[u], m[u], v[u], dw, p.opt.wd, p.opt);
                    p.gW[o[u]] = dw;
                    p.W[o[u]] = w[u]; p.mW[o[u]] = m[u]; p.vW[o[u]] = v[u];
                    stage[rr * SROW + cc] = w[u];
                }
            }
            epi_sync();
            const int64_t k = (int64_t)mt * BM + i, kpad = (K + 63) / 64 * 64;
            if (k < kpad) {                                        // the bf16 copy the next step reads
                float wv[BN];
#pragma unroll
                for (int j = 0; j < BN; ++j) wv[j] = (k < K && n0 + j < H) ? stage[i * SROW + j] : 0.f;
                store_panel_row(p.w16 + (int64_t)e * kpad * train_tc::panels(H) * 128 + nt * kpad * 128, k, wv);
            }
            if (mt == 0 && i < BN && n0 + i < H) {                 // db: the row tiles' partial sums in order
                const int64_t c = n0 + i;
                const int nrt = (int)(p.rpad / BM);
                float db = 0.f;
                for (int t = 0; t < nrt; ++t) db += p.part[((int64_t)e * nrt + t) * H + c];
                const int64_t o = (int64_t)e * H + c;
                p.gb[o] = db;
                float w = p.bb[o], m = p.mb[o], v = p.vb[o];
                adam_elem(w, m, v, db, 0.f, p.opt);
                p.bb[o] = w; p.mb[o] = m; p.vb[o] = v;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 5) tmem_dealloc(tmem, 64);
}

// W [E, K, H] -> W16 panel image: one thread per 8-column chunk of a row
__global__ void pack_w16_kernel(const float* __restrict__ W, int E, int K, int H, uint8_t* __restrict__ w16) {
    const int kpad = (K + 63) / 64 * 64, nch = train_tc::panels(H) * 8;
    const int64_t total = (int64_t)E * kpad * nch;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int q = (int)(t % nch);
        const int64_t k = (t / nch) % kpad, e = t / ((int64_t)nch * kpad);
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int c = q * 8 + j;
            v[j] = (k < K && c < H) ? W[(e * K + k) * H + c] : 0.f;
        }
        uint4 u = {Cvt<1>::pack(v[0], v[1]), Cvt<1>::pack(v[2], v[3]), Cvt<1>::pack(v[4], v[5]), Cvt<1>::pack(v[6], v[7])};
        *reinterpret_cast<uint4*>(w16 + (e * train_tc::panels(H) + q / 8) * kpad * 128 + (k >> 3) * 1024 + panel_off((int)(k & 7), q % 8)) = u;
    }
}

// pens/utils.py:156 into the xs panel image (the arithmetic of scale_in_kernel in train.cu)
__global__ void scale_in_bf16_kernel(const float* __restrict__ x, const float* __restrict__ mu, const float* __restrict__ sig,
                                     int E, int64_t bs, int64_t rpad, int in, uint8_t* __restrict__ xs) {
    const int nch = train_tc::panels(in) * 8;
    const int64_t total = (int64_t)E * rpad * nch;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int q = (int)(t % nch);
        const int64_t r = (t / nch) % rpad, e = t / ((int64_t)nch * rpad);
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int c = q * 8 + j;
            float s = 0.f;
            if (r < bs && c < in) {
                const float xv = x[(e * bs + r) * in + c];
                s = mu ? __fdiv_rn(__fsub_rn(xv, mu[c]), sig[c]) : xv;
            }
            v[j] = s;
        }
        uint4 u = {Cvt<1>::pack(v[0], v[1]), Cvt<1>::pack(v[2], v[3]), Cvt<1>::pack(v[4], v[5]), Cvt<1>::pack(v[6], v[7])};
        *reinterpret_cast<uint4*>(xs + (e * train_tc::panels(in) + q / 8) * rpad * 128 + (r >> 3) * 1024 + panel_off((int)(r & 7), q % 8)) = u;
    }
}

// Loss pass 1 with the arithmetic of loss_pass1_kernel (train.cu), but each block writes its three sums to
// lpart[(e * gridDim.x + block) * 3 + {0,1,2}] instead of adding them atomically: loss pass 2 adds the blocks in
// order, so the step is deterministic.  grid (blocks per member, E), 256 threads.
__global__ void loss_part_bf16_kernel(const float* __restrict__ out, const float* __restrict__ y, const float* __restrict__ mu_out,
                                      const float* __restrict__ sig_out, int64_t bs, int D, int W, int prob,
                                      double* __restrict__ lpart) {
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
    double* q = lpart + ((int64_t)e * gridDim.x + blockIdx.x) * 3;
    if (threadIdx.x == 0) { q[0] = a; q[1] = b; q[2] = c; }
}

// Loss pass 2 with a bf16 output gradient: the per-member loss and d loss / d raw outputs with the arithmetic of
// loss_pass2_kernel (train.cu), written as the G_L panel image, plus the column sums of each 128-row tile.
// grid (panels of W, row tiles, E), 128 threads = the rows of one tile.
__global__ void __launch_bounds__(128) loss_grad_bf16_kernel(const float* __restrict__ out, const float* __restrict__ y,
                                                             const float* __restrict__ mu_out, const float* __restrict__ sig_out,
                                                             int64_t bs, int64_t rpad, int D, int W, int prob, int E,
                                                             const double* __restrict__ lpart, int nblk, float* __restrict__ loss,
                                                             uint8_t* __restrict__ g, float* __restrict__ part) {
    __shared__ float stage[BM * SROW];
    __shared__ double msum[CMBPO_MAX_E][3];
    const int pnl = blockIdx.x, mt = blockIdx.y, e = blockIdx.z, i = threadIdx.x;
    const int64_t n = bs * D;
    if (i < 3 * E) {                                   // member i / 3's sum j = i % 3: its blocks in order
        const int k = i / 3, j = i % 3;
        double t = 0;
        for (int b = 0; b < nblk; ++b) t += lpart[((int64_t)k * nblk + b) * 3 + j];
        msum[k][j] = t;
    }
    __syncthreads();
    const double* sums = &msum[0][0];
    double ts = 0, tq = 0, tl = 0;
    for (int k = 0; k < E; ++k) { ts += sums[k * 3]; tq += sums[k * 3 + 1]; tl += sums[k * 3 + 2]; }
    const float ratio = prob ? (float)(0.05 * ts / tq) : 0.f;
    const float inv_n = 1.0f / (float)n;
    if (pnl == 0 && mt == 0 && i == 0) {
        if (prob) loss[e] = (float)(sums[e * 3] / (double)n + (double)ratio * sums[e * 3 + 1] / (double)n + 0.05 * tl / ((double)n * E));
        else loss[e] = (float)(0.5 * sums[e * 3] / (double)n);
    }
    const int64_t r = (int64_t)mt * BM + i;
    float v[BN];
#pragma unroll
    for (int j = 0; j < BN; ++j) {
        const int c = pnl * BN + j;
        float gv = 0.f;
        if (r < bs && c < W) {
            const int64_t row = ((int64_t)e * bs + r) * W;
            const int d = prob && c >= D ? c - D : c;
            float yt = y[((int64_t)e * bs + r) * D + d];
            if (mu_out) yt = __fdiv_rn(__fsub_rn(yt, mu_out[d]), sig_out[d]);
            const float df = out[row + d] - yt;
            if (!prob) {
                gv = df * inv_n;
            } else if (c < D) {
                gv = 2.0f * df * inv_n;
            } else {
                const float s = df * df, lv = out[row + D + d], ev = expf(lv);
                gv = (2.0f * ratio * (ev - s) * ev + 0.1f * lv) * inv_n;
            }
        }
        v[j] = gv;
        stage[i * SROW + j] = gv;
    }
    store_panel_row(g + (int64_t)e * rpad * train_tc::panels(W) * 128 + pnl * rpad * 128, r, v);
    __syncthreads();
    if (i < BN && pnl * BN + i < W) part[((int64_t)e * gridDim.y + mt) * W + pnl * BN + i] = column_sum(stage, i);
}

int grid_of(cmbpo_ctx* ctx, int64_t n) { return (int)std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * 16); }

template <int USE>
int launch_gemm(cmbpo_ctx* ctx, const GemmParams& p, int n_tiles, int m_tiles) {
    auto kern = train_gemm_kernel<USE>;
    if (!ctx->train_tc_smem_set[USE]) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
        ctx->train_tc_smem_set[USE] = true;
    }
    kern<<<dim3(n_tiles, m_tiles, p.E), NTHREADS, SMEM_BYTES, ctx->stream>>>(p);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

}  // namespace

namespace train_tc {

int pack_w16(cmbpo_ctx* ctx, const float* W, int E, int K, int H, uint8_t* w16) {
    const int64_t total = (int64_t)E * ((K + 63) / 64 * 64) * panels(H) * 8;
    pack_w16_kernel<<<grid_of(ctx, total), 256, 0, ctx->stream>>>(W, E, K, H, w16);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int scale_in(cmbpo_ctx* ctx, const float* x, const float* mu, const float* sig, int E, int64_t bs, int in, uint8_t* xs) {
    const int64_t total = (int64_t)E * rows_pad(bs) * panels(in) * 8;
    scale_in_bf16_kernel<<<grid_of(ctx, total), 256, 0, ctx->stream>>>(x, mu, sig, E, bs, rows_pad(bs), in, xs);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int loss_grad(cmbpo_ctx* ctx, const float* z, const float* y, const float* mu_out, const float* sig_out, int64_t bs,
              int D, int W, int prob, int E, double* lpart, float* loss, uint8_t* g, float* part) {
    const int nblk = loss_blocks(bs, D);
    loss_part_bf16_kernel<<<dim3(nblk, E), 256, 0, ctx->stream>>>(z, y, mu_out, sig_out, bs, D, W, prob, lpart);
    loss_grad_bf16_kernel<<<dim3(panels(W), row_tiles(bs), E), 128, 0, ctx->stream>>>(z, y, mu_out, sig_out, bs, rows_pad(bs), D, W,
                                                                                     prob, E, lpart, nblk, loss, g, part);
    ctx->launches += 2;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int forward(cmbpo_ctx* ctx, int E, int64_t bs, int K, int H, const uint8_t* a, const uint8_t* w16, const float* b,
            int act, float* z, uint8_t* h) {
    GemmParams p = {};
    p.E = E; p.nk = panels(K); p.bs = bs; p.rpad = rows_pad(bs); p.K = K; p.H = H;
    p.a = a; p.a_panel = p.rpad * 128; p.a_member = p.a_panel * panels(K); p.a_npanels = panels(K);
    p.b = w16; p.b_panel = (int64_t)((K + 63) / 64 * 64) * 128; p.b_member = p.b_panel * panels(H);
    p.bias = b; p.act = act; p.z = z; p.h = h;
    return launch_gemm<FWD>(ctx, p, panels(H), row_tiles(bs));
}

int data_grad(cmbpo_ctx* ctx, int E, int64_t bs, int K, int H, const uint8_t* g, const uint8_t* w16,
              const float* z_prev, int act_prev, uint8_t* g_prev, float* part_prev) {
    GemmParams p = {};
    p.E = E; p.nk = panels(H); p.bs = bs; p.rpad = rows_pad(bs); p.K = K; p.H = H;
    p.a = g; p.a_panel = p.rpad * 128; p.a_member = p.a_panel * panels(H); p.a_npanels = panels(H);
    p.b = w16; p.b_panel = (int64_t)((K + 63) / 64 * 64) * 128; p.b_member = p.b_panel * panels(H);
    p.z_prev = z_prev; p.act = act_prev; p.g_out = g_prev; p.part_out = part_prev;
    return launch_gemm<DGRAD>(ctx, p, panels(K), row_tiles(bs));
}

int weight_grad_adam(cmbpo_ctx* ctx, int E, int64_t bs, int K, int H, const uint8_t* a, const uint8_t* g,
                     const float* part, float* W, float* mW, float* vW, float* gW, float* b, float* mb, float* vb,
                     float* gb, uint8_t* w16, Adam opt) {
    GemmParams p = {};
    p.E = E; p.nk = (int)((bs + BK - 1) / BK); p.bs = bs; p.rpad = rows_pad(bs); p.K = K; p.H = H;
    p.a = a; p.a_panel = p.rpad * 128; p.a_member = p.a_panel * panels(K); p.a_npanels = panels(K);
    p.b = g; p.b_panel = p.rpad * 128; p.b_member = p.b_panel * panels(H);
    p.part = part; p.W = W; p.mW = mW; p.vW = vW; p.gW = gW; p.bb = b; p.mb = mb; p.vb = vb; p.gb = gb; p.w16 = w16;
    p.opt = opt;
    return launch_gemm<WGRAD>(ctx, p, panels(H), (K + BM - 1) / BM);
}

}  // namespace train_tc
