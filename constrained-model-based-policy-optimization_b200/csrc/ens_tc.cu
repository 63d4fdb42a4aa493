// K1 on the tensor cores: the 3-layer ensemble MLP chain  X -> act(X W0+b0) -> act(. W1+b1) -> . W2+b2
// for one 128-row tile per CTA and all E members, with tcgen05.mma (kind::f16, fp32 accumulators in
// TMEM).  Hidden activations never leave the SM and never touch shared memory: they live in TENSOR
// MEMORY as the A operand of the next layer (tcgen05.mma with A from TMEM), which leaves almost all
// of shared memory to the rings of weight tiles streamed from L2 by the bulk-copy engine (5 x 32 KB
// for layers 0/1, 2 x 24 KB for layer 2; pre-swizzled tile images, plain 1-D cp.async.bulk, no
// tensor maps).
//
//   TMEM columns (512):   H1  [0, HD/2)      layer-0 output, 16-bit packed 2/column  (A of layer 1)
//                         D   2 x 64         fp32 accumulator chunks (double buffered)
//                         H2  1-2 x 32       layer-1 output chunk, 16-bit packed       (A of layer 2)
//                         OUT NP             layer-2 accumulator (all chunks accumulate into it)
//   layer 0   D chunk[128 x 64] = XA(smem) x W0 chunk           (K = in_dim padded to 16)
//             epilogue: +bias, act -> 16-bit -> tcgen05.st into H1
//   layer 1   D chunk = sum over 64-wide K panels  H1[kp](tmem) x W1[kp, chunk]
//             epilogue: +bias, act -> 16-bit -> tcgen05.st into an H2 buffer
//   layer 2   OUT[128 x NP] += H2(tmem) x W2[chunk rows, :]
//             epilogue: +b2 -> raw outputs (fp32) to global
//
// Warp roles (640 threads): warp 0 = layer-0/1 weight producer, warp 1 = layer-0/1 MMA issuer, warp 2 =
// TMEM allocator + layer-2 MMA issuer, warp 3 = layer-2 weight producer (setmaxnreg 32), warps 4-19 =
// four epilogue warpgroups (setmaxnreg 112; thread <-> row <-> TMEM lane; a pair of warpgroups owns
// one accumulator buffer, each warpgroup 32 of the chunk's 64 columns).  Work unit = (row tile,
// member), or (row tile, group of 4 narrow members) in grouped mode.  Wide ordinary ensembles run as CLUSTER PAIRS
// (template parameter CL = 2): two CTAs work on the same member and multicast one copy of its weights into both
// rings (see the comment at the kernel).
//
// Replaces models/pens/fc.py:74-95 x3 + the input scaler of models/pens/utils.py:156 (fused into the
// XA load).  The output scaler / exp are applied by the consumer (ens_head_kernel or the rollout row
// math) exactly as on the fp32 path.
#include <cstring>
#include "tc_common.cuh"
#include "step_common.cuh"

using namespace tc;

namespace {

constexpr int NTHREADS = 640;    // 4 control warps + 16 epilogue warps
constexpr int TILE = 8192;        // [64 neurons x 64 k x 2 B] weight tile
constexpr int STAGE = 4 * TILE;   // main-ring stage: up to 4 consecutive tiles (one mbarrier wait per 16 MMAs)
constexpr int NSM = 5;            // main ring depth (160 KB)
constexpr int W2SLOT = 16384;     // layer-2 ring slot: the W2 tiles of CPS consecutive chunks (NP <= 128: >= 1 chunk)
constexpr int NS2 = 2;
constexpr int BIAS_SLOT = 4096;   // per-unit hidden biases [b0 | b1] (<= 2 x 512 floats), double buffered
constexpr int XA_BYTES = 16384;   // [128 rows x 64 k x 2 B]

struct Stage {        // one weight tile image in the packed stream
    int layer, n0, k0, rows, member;   // member: index inside a group (0 for ordinary nets)
    unsigned long long off;
};

struct TcParams {
    const uint8_t* wmain; unsigned long long main_bytes;   // per member: layer-0 + layer-1 tiles
    const uint8_t* w2; unsigned long long w2_bytes;        // per member: layer-2 tiles
    const float* bias; int bias_stride;
    int E, K0, KS0, Nout, NP, parts, cps;        // parts = 2 when NP > 64; cps = chunks per W2 slot
    int fold;                                    // layer-0 bias rides in the GEMM (XA columns K0, K0+1 = 1)
    const float* x; long long N; int ldx;
    const long long* n_dev;                      // optional: live row count on the device (<= N)
    const float *mu_in, *sig_in;
    float* out; long long out_member_stride;   // out[e*stride + row*Nout + c]
    int ntiles;
    int member_act[CMBPO_MAX_E];   // ACT == 0 kernels (merged nets): hidden activation per member
    FusedStep fz;              // FUSE kernels only: the rollout step around the GEMM chain (step_common.cuh)
};

// barrier indices
enum { W_FULL = 0, W_EMPTY = NSM, W2_FULL = 2 * NSM, W2_EMPTY = 2 * NSM + NS2, D_FULL = 2 * NSM + 2 * NS2,
       D_EMPTY = D_FULL + 2, H1_FULL = D_FULL + 4, H2_FULL = D_FULL + 5, H2_EMPTY = D_FULL + 7,
       OUT_FULL = D_FULL + 9, OUT_EMPTY = D_FULL + 10, X_FULL = D_FULL + 11, B_FULL = D_FULL + 12,
       B_EMPTY = D_FULL + 14, NBAR = D_FULL + 16 };
// wide-output deep kernels (WO, no H2 buffers): "last-hidden chunk j drained", j < 4, in the four H2 barriers
constexpr int HL_FULL = H2_FULL;
static_assert(H2_EMPTY == H2_FULL + 2, "HL_FULL spans the H2_FULL and H2_EMPTY pairs");
constexpr int SMEM_W2 = XA_BYTES + NSM * STAGE;
constexpr int SMEM_BIAS = SMEM_W2 + NS2 * W2SLOT;
constexpr int SMEM_IN_BYTES = 512;   // input scaler: mu[64] | sigma[64]
constexpr int SMEM_BAR = SMEM_BIAS + 2 * BIAS_SLOT + SMEM_IN_BYTES;
constexpr int SMEM_TOTAL = SMEM_BAR + NBAR * 8 + 16;
// FUSE kernels (the rollout step fused around the GEMM chain): the layer-2 ring shrinks to 2 x 12 KB (a
// 2 x 8 KB ring measured the same as 2 x 24 KB) and the freed shared memory stages the row math:
//   stage  12 KB   kl, epv per (obs dimension, row) of one pass of RP rows (RP = 64 / 32 by obs dim)
//   misc    5 KB   per-row member / path / state / non-finite flag, the 4 next-state coordinates the statics
//                  read, output-scaler vectors, log_std, elite list, the "last arriver" flag
constexpr int W2SLOT_F = 12288;
constexpr int FZ_STAGE = 12288, FZ_MISC = 5120;
constexpr int SMEM_BIAS_F = SMEM_W2 + NS2 * W2SLOT_F;
constexpr int SMEM_BAR_F = SMEM_BIAS_F + 2 * BIAS_SLOT + SMEM_IN_BYTES;
constexpr int SMEM_FZ = SMEM_BAR_F + NBAR * 8 + 16;
constexpr int SMEM_TOTAL_F = SMEM_FZ + FZ_STAGE + FZ_MISC;
static_assert(SMEM_FZ % 16 == 0 && SMEM_TOTAL_F + 1024 <= 232448, "fused shared-memory budget");

struct FzSmem {          // views into the misc area
    float *kl, *epv;                 // [O][RP]
    int *member, *path;              // [128]
    int* nonfin;                     // [128]
    float* spec;                     // [4][128]: next_obs[0], [2], [3], [O-1]
    float *sig, *mu, *l2s;           // [64] output scaler (pens/utils.py:167,187)
    float* log_std;                  // [32]
    int* elite;                      // [8]
    unsigned char* state;            // [128]
    int* flag;
};
__device__ __forceinline__ FzSmem fz_views(uint8_t* base) {
    FzSmem m;
    m.kl = reinterpret_cast<float*>(base);
    m.epv = nullptr;                 // set per launch geometry: kl + O * RP
    uint8_t* q = base + FZ_STAGE;
    m.member = reinterpret_cast<int*>(q); q += 512;
    m.path = reinterpret_cast<int*>(q); q += 512;
    m.nonfin = reinterpret_cast<int*>(q); q += 512;
    m.spec = reinterpret_cast<float*>(q); q += 2048;
    m.sig = reinterpret_cast<float*>(q); q += 256;
    m.mu = reinterpret_cast<float*>(q); q += 256;
    m.l2s = reinterpret_cast<float*>(q); q += 256;
    m.log_std = reinterpret_cast<float*>(q); q += 128;
    m.elite = reinterpret_cast<int*>(q); q += 32;
    m.state = q; q += 128;
    m.flag = reinterpret_cast<int*>(q); q += 16;
    return m;                        // 4656 B <= FZ_MISC
}

__device__ __forceinline__ void epi_bar() {      // named barrier 1: the 512 epilogue threads
    asm volatile("bar.sync 1, 512;" ::: "memory");
}

// ---- the rollout step's row math for one finished row tile (all E members' outputs sit in the L2
// scratch), run by the 512 epilogue threads of the CTA that delivered the tile's last member.
// Same phases and literally the same per-row functions as rollout_step_kernel (rollout.cu):
//   0  one thread per row: elite member, carried per-path scalars
//   1  one thread per (obs dim, row), lanes along rows (coalesced scratch reads): member statistics, KL
//   2  one thread per row: ordered sums over dims (numpy order), statics, sampler rules, per-step scalars
//   3  one thread per (row, dim), lanes along dims (coalesced buffer writes): next state of the chosen
//      member recomputed (bit-identical), obs / next_obs / act / mu rows, carried state
__device__ __forceinline__ void fused_rows(const FusedStep& f, const FzSmem& sm, int tile, long long n_rows, int etid) {
    const int O = f.O, A = f.A, W = 2 * f.c.D, t = f.rules.t, sh = f.rp_shift, RP = 1 << sh;
    const float* tbase = f.raw_tiles + (size_t)tile * f.c.E * W * 128;
    EnvRowCfg c = f.c;
    c.sig_out = sm.sig; c.mu_out = sm.mu; c.l2s_out = sm.l2s; c.elite = sm.elite;
    float* s_kl = sm.kl;
    float* s_epv = sm.kl + O * RP;
    const int lane = etid & 31;
    for (int r0 = 0; r0 < 128; r0 += RP) {
        const long long base = (long long)tile * 128 + r0;
        if (base >= n_rows) break;                                   // uniform
        float pf_v = 0.f, pf_vc = 0.f, pf_logp = 0.f;
        double pf_dkl = 0.0, pf_ret = 0.0, pf_cost = 0.0;
        if (etid < RP) {
            const long long r = base + etid;
            int member = -1, path = -1;
            if (r < n_rows) {
                path = f.row_path ? f.row_path[r] : (int)r;
                if (f.rules.alive[path]) {
                    const int pos = f.elite_pos ? f.elite_pos[path] : philox_elite_pos(f.seed, f.path_base + path, t, f.n_elite);
                    member = sm.elite[pos];
                    pf_v = f.vrow[r]; pf_vc = f.vcrow[r]; pf_logp = f.logp[r];
                    pf_dkl = f.rules.b.cum_dkl[path]; pf_ret = f.rules.b.path_return[path]; pf_cost = f.rules.b.path_cost[path];
                }
            }
            sm.member[etid] = member; sm.path[etid] = path; sm.state[etid] = 0; sm.nonfin[etid] = 0;
        }
        epi_bar();
        const int NI = RP * O;
        for (int idx = etid; idx < NI; idx += 512) {
            const int rr = idx & (RP - 1), dim = idx >> sh;
            const int member = sm.member[rr];
            if (member < 0) continue;
            const long long pth = sm.path[rr];
            float eps = 1.0f;
            if (!c.deterministic)
                eps = f.state_eps ? f.state_eps[pth * O + dim] : philox_normal(f.seed, f.path_base + pth, t, RNG_STREAM_STATE, dim);
            RawTile raw(tbase, W, r0 + rr);
            const EnvDimOut d = env_dim<7, true>(c, raw, dim, member, f.cur_obs[(base + rr) * O + dim], eps);
            s_kl[idx] = d.kl; s_epv[idx] = d.epv;
            if (!isfinite(d.nx)) sm.nonfin[rr] = 1;
            if (dim == 0) sm.spec[rr] = d.nx;
            if (dim == 2) sm.spec[128 + rr] = d.nx;
            if (dim == 3) sm.spec[256 + rr] = d.nx;
            if (dim == O - 1) sm.spec[384 + rr] = d.nx;
        }
        epi_bar();
        double st0 = 0.0, st1 = 0.0, st2 = 0.0, st3 = 0.0;
        if (etid < RP) {
            const int member = sm.member[etid];
            if (member >= 0) {
                const long long pth = sm.path[etid];
                RawTile raw(tbase, W, r0 + etid);
                const float ks = np_sum_strided(s_kl + etid, O, RP), es = np_sum_strided(s_epv + etid, O, RP);
                const EnvRowOut o = env_row_core<true>(c, raw, member, ks, es, sm.nonfin[etid] == 0, sm.spec[etid],
                                                       sm.spec[128 + etid], sm.spec[256 + etid], sm.spec[384 + etid]);
                RowCarry pf;
                pf.v = pf_v; pf.vc = pf_vc; pf.logp = pf_logp; pf.dkl = pf_dkl; pf.ret = pf_ret; pf.cost = pf_cost;
                sm.state[etid] = (unsigned char)step_row_commit(f.rules, pth, o, pf, st0, st1, st2, st3);
            }
            // per-step statistics: one reduction per warp of row threads, four REDs per warp
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                st0 += __shfl_down_sync(0xffffffffu, st0, off); st1 += __shfl_down_sync(0xffffffffu, st1, off);
                st2 += __shfl_down_sync(0xffffffffu, st2, off); st3 += __shfl_down_sync(0xffffffffu, st3, off);
            }
            if (lane == 0 && st0 != 0.0) {
                double* ss = f.rules.b.step_stats + (long long)t * 4;
                atomicAdd(ss + 0, st0); atomicAdd(ss + 1, st1); atomicAdd(ss + 2, st2); atomicAdd(ss + 3, st3);
            }
        }
        epi_bar();
        for (int idx = etid; idx < NI; idx += 512) {
            const int rr = idx / O, dim = idx - rr * O;
            if (sm.state[rr] != 1) continue;
            const int member = sm.member[rr];
            const long long pth = sm.path[rr], row = (long long)t * f.rules.B + pth;
            float eps = 1.0f;
            if (!c.deterministic)
                eps = f.state_eps ? f.state_eps[pth * O + dim] : philox_normal(f.seed, f.path_base + pth, t, RNG_STREAM_STATE, dim);
            RawTile raw(tbase, W, r0 + rr);
            const float ob = f.cur_obs[(base + rr) * O + dim];
            const float nx = env_dim_nx<true>(c, raw, dim, member, ob, eps);
            if (!f.rules.no_store) {
                f.rules.b.obs[row * O + dim] = ob;
                f.rules.b.nextobs[row * O + dim] = nx;
            }
            f.cur_obs[(base + rr) * O + dim] = nx;                 // model_sampler.py:350
        }
        if (!f.rules.no_store)
        for (int idx = etid; idx < RP * A; idx += 512) {
            const int rr = idx / A, i = idx - rr * A;
            if (sm.state[rr] != 1) continue;
            const long long pth = sm.path[rr], row = (long long)t * f.rules.B + pth;
            f.rules.b.act[row * A + i] = f.pi[(base + rr) * A + i];
            f.rules.b.mu[row * A + i] = f.mu[(base + rr) * A + i];
        }
        epi_bar();                                                   // the staging is reused by the next pass / tile
    }
}


// 32 accumulator columns of this thread's row -> (+bias), act -> 16-bit pairs -> 16 TMEM columns.
// The accumulator buffer is released (`d_empty`) as soon as the values sit in registers; the
// destination is only waited for (`dst_free`, 0 = none) right before the store.
//
// Swish members are packed with their hidden-layer weights and biases HALVED (exact in 16 bits), so the
// accumulator already holds t = x/2 and swish(x) = t + t tanh t needs one MUFU and one FFMA.  `bias`
// points at this warp's 32 biases in shared memory (every lane reads the same address: a broadcast
// LDS.128 per four elements; the earlier per-element SHFL of a lane-held bias shared the MIO queue with
// the MUFU instructions) or is null when the bias rides in the GEMM (layer 0, see `fold`).  ACT == 0: the
// activation is a per-member runtime value (merged policy ensemble), swish when `rt_swish`, else tanh.
template <int FMT, int ACT>
__device__ __forceinline__ void drain32(uint32_t d_addr, const float* bias, uint32_t dst_addr,
                                        uint32_t d_empty, uint32_t dst_free, uint32_t dst_parity,
                                        bool rt_swish = false) {
    uint32_t r[32];
    tmem_ld32(d_addr, r);
    tmem_ld_wait();
    tc_fence_before();
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive_a(d_empty);
    uint32_t q[16];
    float v[32];
    if (bias) {
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
            const float4 b = *reinterpret_cast<const float4*>(bias + i);
            v[i] = __uint_as_float(r[i]) + b.x; v[i + 1] = __uint_as_float(r[i + 1]) + b.y;
            v[i + 2] = __uint_as_float(r[i + 2]) + b.z; v[i + 3] = __uint_as_float(r[i + 3]) + b.w;
        }
    } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
    }
#pragma unroll
    for (int i = 0; i < 32; ++i) {
        if (ACT == 0) {          // per-member run-time activation, ONE copy of the code: both forms from one MUFU, then a select
            const float r = tanh_approx(v[i]);
            const float sw = fmaf(v[i], r, v[i]);
            v[i] = rt_swish ? sw : r;
        } else {
            v[i] = (ACT == CMBPO_ACT_SWISH) ? swish_half(v[i]) : tanh_approx(v[i]);
        }
    }
#pragma unroll
    for (int c = 0; c < 16; ++c) q[c] = Cvt<FMT>::pack(v[2 * c], v[2 * c + 1]);
    if (dst_free) { mbar_wait_a(dst_free, dst_parity); tc_fence_after(); }
    tmem_st16(dst_addr, q);
    tmem_st_wait();
    tc_fence_before();
}

// G > 1: GROUPED mode for narrow members (width HD/G): G members form one unit whose layer 0 is one
// dense HD-wide layer (all chunks share the XA panel) and whose layers 1-2 are block diagonal (chunk j
// belongs to member j / (NC/G), uses only that member's K panels and accumulates into that member's
// OUT block).  A narrow net processed alone is a serial chain of tiny MMAs and drains; grouped, the
// chunks of G members flow through the same double-buffered pipeline as one wide member.
// NMID > 0: DEEPER networks (2 + NMID hidden layers, e.g. the reference's code default (200,200,200,200),
// algorithms/cmbpo.py:54): a second hidden-activation buffer HB in tensor memory, the hidden layers ping-pong
// between H1 and HB (layer 0 writes H1; middle layer i reads buffer (i-1)&1 and writes buffer i&1; the last
// hidden layer reads buffer NMID&1 and feeds H2 / layer 2 as before).  Needs 2 x HD/2 + 192 + NP <= 512 columns:
// padded width <= 256 and NP <= 64.  No extra barriers: the tensor pipe executes in order, so by the time a
// chunk's accumulator is handed to the epilogue every MMA that read the buffer it is about to overwrite has
// finished; H1_FULL simply completes once per hidden layer instead of once per unit.
// WO (deep nets with 64 < NP <= 128): there is no room for H2 next to a 128-column OUT, so the last hidden layer
// writes its whole output into the idle hidden buffer, like a middle layer (it reads buffer NMID&1 and writes
// buffer LAST = (NMID+1)&1), and layer 2 reads its A operand straight from there, one N = NP MMA per K step:
//   H1 [0,128)   D [128,256)   HB [256,384)   OUT [512-NP,512) within [384,512)
// The W2 stream is unchanged: the two NP/2-row tiles of a chunk are, back to back, one NP-row tile.  The layer-2
// issuer takes K panel j as soon as last-hidden chunk j is drained (HL_FULL + j, once per unit).  The buffers:
//  * the last-hidden drains overwrite buffer LAST only after everything that read it earlier: the layer before
//    (the D_FULL of a last-hidden chunk follows it in the layer-0/1 issuer's order) and the previous unit's layer 2
//    (see the next point);
//  * the next unit writes buffer LAST again -- at NMID = 1 (LAST = H1) in its layer-0 drains, at NMID = 2
//    (LAST = HB) in its first middle-layer drains.  Those stores must wait for this unit's layer-2 MMAs, which a
//    different thread issues (no tensor-pipe order with the layer-0/1 issuer's commits).  At NMID = 2 they follow
//    the deferred OUT epilogue, whose OUT_FULL wait is exactly that; at NMID = 1 the layer-0 drains come first, so
//    each epilogue warp's first layer-0 store of a unit waits for the previous unit's OUT_FULL itself.  This also
//    keeps the epilogue less than a unit ahead of the layer-2 issuer, which makes one HL_FULL phase per unit exact.
// CL == 2: the CTAs run as CLUSTER PAIRS that stream ONE copy of the weights from L2: both CTAs of a pair work on
// the same member (two neighbouring row tiles), each fetches half of every main-ring stage and MULTICASTS it into
// both CTAs' rings.  Why: the layer-1 phase needs a 2 KB weight tile per 32-cycle MMA = 64 B/clk per SM, and 148 SMs
// x 64 B/clk is more than the L2 slices deliver (~6300 B/clk chip-wide = 42 B/clk per SM, B300_MICROARCH.md):
// the phase ran at ~47 cycles per MMA.  Everything else (MMAs, tensor memory, epilogue) stays per CTA (cta_group::1);
// only a ring slot's release is a pair-wide event (both issuers commit to both CTAs' W_EMPTY barriers).
template <int HD, int FMT, int ACT, int G, bool FUSE, int NMID = 0, int CL = 1, bool WO = false>
__global__ void __launch_bounds__(NTHREADS, 1) ens_mlp3_tc_kernel(const TcParams p) {
    static_assert(CL == 1 || (CL == 2 && G == 1 && !FUSE), "cluster pairs: ordinary ensembles only");
    static_assert(!FUSE || G == 1, "the fused step kernel exists for ordinary (ungrouped) ensembles");
    static_assert(NMID == 0 || (HD <= 256 && G == 1 && !FUSE), "deep variant: width <= 256, ungrouped");
    static_assert(!WO || (NMID > 0 && HD == 256 && CL == 1), "wide-output variant: deep nets at padded width 256");
    constexpr int W2S = FUSE ? W2SLOT_F : W2SLOT;          // layer-2 ring slot bytes
    constexpr int NC = HD / 64;                     // 64-column chunks of a hidden layer
    constexpr int KP = HD / 64 / G;                 // 64-wide K panels of layer 1 (per member)
    constexpr int CPM = NC / G;                     // chunks per member
    constexpr int TPS = KP < 4 ? KP : 4;            // layer-1 tiles (K panels) per main-ring stage
    constexpr int G0 = NC < 4 ? NC : 4;             // layer-0 chunk tiles per main-ring stage
    constexpr uint32_t COL_H1 = 0, COL_D = HD / 2, COL_H2 = COL_D + 128;
    constexpr uint32_t COL_HB = WO ? COL_H2 : COL_H2 + 64;     // second hidden-activation buffer (NMID > 0 only)
    constexpr int NHID = 1 + NMID;                 // HD x HD layers: NMID middle ones + the last hidden layer
    constexpr uint32_t COL_LAST = ((NMID + 1) & 1) ? COL_HB : COL_H1;     // WO: the last hidden layer's output
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sXA = smem;
    uint8_t* sW = smem + XA_BYTES;
    uint8_t* sW2 = smem + SMEM_W2;
    float* sBias = reinterpret_cast<float*>(smem + (FUSE ? SMEM_BIAS_F : SMEM_BIAS));
    float* sIn = sBias + 2 * BIAS_SLOT / 4;
    constexpr int BAR_OFF = FUSE ? SMEM_BAR_F : SMEM_BAR;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + BAR_OFF);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + BAR_OFF + NBAR * 8);

    // Warp roles: 0 = main weight producer, 1 = layer-0/1 MMA issuer, 2 = TMEM allocator + layer-2 MMA
    // issuer, 3 = W2 producer, 4-19 = epilogue (four warpgroups).  A warp may only touch the TMEM lane
    // quarter (warp id % 4), which is also its sub-core, so every sub-core hosts four epilogue warps.
    const int hw_warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int warp = hw_warp;                                  // role id: 0-3 control, 4-19 epilogue
    const int nh2 = (p.parts == 1) ? 2 : 1;                    // H2 buffers (TMEM budget)
    const uint32_t col_out = 512u - (uint32_t)(p.NP * G);      // OUT occupies the top G*NP columns
    const int NPp = p.NP / p.parts;
    const uint32_t w2_chunk_bytes = (uint32_t)p.NP * 128u;     // all parts of one chunk
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < NSM; ++i) { mbar_init(bar + W_FULL + i, 1); mbar_init(bar + W_EMPTY + i, CL); }
        for (int i = 0; i < NS2; ++i) { mbar_init(bar + W2_FULL + i, 1); mbar_init(bar + W2_EMPTY + i, 1); }
        for (int i = 0; i < 2; ++i) {
            mbar_init(bar + D_FULL + i, 1); mbar_init(bar + D_EMPTY + i, 8);
            mbar_init(bar + H2_FULL + i, 8); mbar_init(bar + H2_EMPTY + i, WO ? 8 : 1);    // WO: HL_FULL + 2 + i
        }
        mbar_init(bar + H1_FULL, 8 * NC);
        mbar_init(bar + OUT_FULL, 1); mbar_init(bar + OUT_EMPTY, 16);
        mbar_init(bar + X_FULL, 4);
        for (int i = 0; i < 2; ++i) { mbar_init(bar + B_FULL + i, 1); mbar_init(bar + B_EMPTY + i, 16); }
        fence_barrier_init();
    }
    if (warp == 2) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (CL == 2) cluster_sync_all();      // the peer's barriers are initialised before anything is sent to them
    const uint32_t cta_rank = (CL == 2) ? cluster_ctarank() : 0u;
    // The CTA owns all 512 columns, so the allocation can only start at lane 0 / column 0.  Treating
    // the base as the constant 0 keeps every MMA operand address in uniform registers (a base read
    // back from shared memory forces a per-instruction R2UR waterfall, ~100 cycles per MMA).
    if (*tmem_slot != 0u) __trap();     // (no printf: a device-side call constrains the hot loops' registers)
    constexpr uint32_t tmem = 0u;
    // Work unit = (row tile, member): the ntiles*E units are split into contiguous, equal ranges, one
    // per CTA, so the last wave is balanced to within one member (a tile-granular split leaves the
    // last of ceil(782/148) = 6 rounds 72% empty), and neighbouring CTAs start on different members,
    // which spreads the weight streaming over E x more L2 addresses.
    const int n_groups = (p.E + G - 1) / G;         // E itself when G == 1
    // the live row count may sit in device memory (alive-row compaction of the rollout): rows beyond
    // it are not computed; strides still use the allocated N
    const long long n_rows = p.n_dev ? *p.n_dev : p.N;
    // CL == 2: a unit is (PAIR of row tiles, member), split over the cluster pairs; CTA r of a pair takes tile 2 tp + r
    // (an odd tile count leaves the last pair one tile without rows: it runs the protocol and stores nothing)
    const long long n_units = ((n_rows + 128 * CL - 1) / (128 * CL)) * n_groups;      // < 2^31 (checked by the host)
    const long long w_idx = blockIdx.x / CL, w_cnt = gridDim.x / CL;
    const int u0 = (int)(n_units * w_idx / w_cnt), u1 = (int)(n_units * (w_idx + 1) / w_cnt);
#define CMBPO_TILE_OF(u) ((int)((u) / n_groups) * CL + (int)cta_rank)

    // (The pool is the CTA's own allocation of 640 x 96 registers: the 128 x (96 - 32) released by the
    // control warpgroup are exactly the 4 x 128 x 16 the epilogue warpgroups request; asking for more
    // blocks setmaxnreg.inc forever.  32 is enough for the control warps: their MMA / copy operands live
    // in uniform registers.)
    // Register re-balancing (per warpgroup): the control warpgroup needs few registers, the epilogue
    // warps need enough to keep all 32 element chains of a drain in flight (at the 96 of the launch
    // bound ptxas serialises them through one temporary: ~2000 instead of ~500 cycles per drain).
    if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 32;");
    if (warp == 0) {
        // ===== main weight producer: layer-0 and layer-1 tiles, 32 KB per stage =====
        uint32_t s = 0, ph = 0;
        for (int u = u0; u < u1; ++u) {
            {
                const int e = (int)(u % n_groups);
                const uint8_t* src = p.wmain + (unsigned long long)e * p.main_bytes;
                auto push = [&](uint32_t bytes) {
                    mbar_wait(bar + W_EMPTY + s, ph ^ 1);
                    if (elect_one()) {
                        mbar_expect_tx(bar + W_FULL + s, bytes);
                        if (CL == 2)      // my half of the stage, into both CTAs' rings; the peer sends the other half
                            bulk_g2s_mc(sW + s * STAGE + cta_rank * (bytes / 2), src + cta_rank * (bytes / 2), bytes / 2,
                                        bar + W_FULL + s, (uint16_t)3);
                        else
                            bulk_g2s(sW + s * STAGE, src, bytes, bar + W_FULL + s);
                    }
                    __syncwarp();
                    src += bytes;
                    if (++s == NSM) { s = 0; ph ^= 1; }
                };
                for (int j0 = 0; j0 < NC; j0 += G0) push(G0 * TILE);
                for (int lyr = 0; lyr < NHID; ++lyr)
                    for (int j = 0; j < NC; ++j)
                        for (int kq = 0; kq < KP / TPS; ++kq) push(TPS * TILE);
            }
        }
    } else if (warp == 3) {
        // ===== layer-2 weight producer: the W2 tiles of `cps` consecutive chunks per slot =====
        uint32_t s2 = 0, ph2 = 0, mb = 0;
        for (int u = u0; u < u1; ++u, ++mb) {
            {
                const int e = (int)(u % n_groups);
                {   // hidden-layer biases [b0 | b1] of this unit -> bias buffer (mb & 1)
                    mbar_wait(bar + B_EMPTY + (mb & 1), ((mb >> 1) & 1) ^ 1);
                    if (elect_one()) {
                        mbar_expect_tx(bar + B_FULL + (mb & 1), (1 + NHID) * HD * 4);
                        bulk_g2s(sBias + (mb & 1) * (BIAS_SLOT / 4), p.bias + (long long)e * p.bias_stride, (1 + NHID) * HD * 4,
                                 bar + B_FULL + (mb & 1));
                    }
                    __syncwarp();
                }
                const uint8_t* src = p.w2 + (unsigned long long)e * p.w2_bytes;
                for (int j0 = 0; j0 < NC; j0 += p.cps) {
                    const int nchunks = (NC - j0) < p.cps ? (NC - j0) : p.cps;
                    const uint32_t bytes = (uint32_t)nchunks * w2_chunk_bytes;
                    mbar_wait(bar + W2_EMPTY + s2, ph2 ^ 1);
                    if (elect_one()) {
                        mbar_expect_tx(bar + W2_FULL + s2, bytes);
                        bulk_g2s(sW2 + s2 * W2S, src, bytes, bar + W2_FULL + s2);
                    }
                    __syncwarp();
                    src += bytes;
                    if (++s2 == NS2) { s2 = 0; ph2 ^= 1; }
                }
            }
        }
    } else if (warp == 2) {
        // ===== layer-2 MMA issuer: OUT(member) += H2[chunk] x W2[rows of the chunk] =====
        // A warp of its own: the bookkeeping of a partial (three barrier waits, two commits) costs the
        // issuing thread ~1000 cycles per chunk, which on the layer-1 issuer's instruction stream was
        // the kernel's critical path.  The two issuers only meet in the tensor pipe.
        const uint32_t idesc_o = idesc_f16(FMT, WO ? p.NP : NPp);
        const uint64_t dW2 = smem_desc_sw128(smem_u32(sW2));
        uint32_t s2 = 0, ph2 = 0, c1 = 0, m = 0;
        for (int u = u0; u < u1; ++u) {
            int jin = 0;
            for (int jj = 0; jj < NC; ++jj) {
                // barrier pair = chunk parity (one per epilogue pair), also when H2 is single buffered:
                // every waiter then sees consecutive phases of "its" barrier and the parity test is exact
                const uint32_t hbar = c1 & 1, hn = c1 >> 1, hb = (nh2 == 2) ? hbar : 0;
                if (jin == 0) mbar_wait(bar + W2_FULL + s2, ph2);
                if (jj == 0) mbar_wait(bar + OUT_EMPTY, (m & 1) ^ 1);
                if constexpr (WO) mbar_wait(bar + HL_FULL + jj, m & 1);
                else mbar_wait(bar + H2_FULL + hbar, hn & 1);
                tc_fence_after();
                const bool last_in_slot = (jin == p.cps - 1) || (jj == NC - 1);
                if (elect_one()) {
                    if constexpr (WO) {      // K panel jj of the last hidden layer x the chunk's NP-row W2 tile
                        const uint64_t dB = dW2 + (uint64_t)((s2 * W2S + jin * p.NP * 128) >> 4);
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks)
                            mma_f16_ts(tmem + col_out, tmem + COL_LAST + jj * 32 + ks * 8, dB + 2 * ks, idesc_o,
                                       !(jj == 0 && ks == 0));
                    } else {
                    for (int q = 0; q < p.parts; ++q) {
                        const uint64_t dB = dW2 + (uint64_t)((s2 * W2S + (jin * p.parts + q) * NPp * 128) >> 4);
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks)
                            mma_f16_ts(tmem + col_out + (jj / CPM) * p.NP + q * NPp, tmem + COL_H2 + hb * 32 + ks * 8,
                                       dB + 2 * ks, idesc_o, !(jj % CPM == 0 && ks == 0));
                    }
                    mma_commit(bar + H2_EMPTY + hbar);
                    }
                    if (last_in_slot) mma_commit(bar + W2_EMPTY + s2);
                    if (jj == NC - 1) mma_commit(bar + OUT_FULL);
                }
                __syncwarp();
                if (last_in_slot) { jin = 0; if (++s2 == NS2) { s2 = 0; ph2 ^= 1; } } else ++jin;
                ++c1;
            }
            ++m;
        }
    } else if (warp == 1) {
        // ===== layer-0/1 MMA issuer.  Wide members (G == 1): ONE elected thread runs the whole loop, waits
        // included, so that no warp-level election / reconvergence sits between two batches of MMAs
        // (-6% on the 512-wide ensemble).  Grouped narrow members have short batches and are paced by
        // the drains; there the warp-uniform loop with a per-batch election measured 5% faster. =====
                constexpr bool SINGLE = (G == 1);
        const uint32_t idesc_h = idesc_f16(FMT, 64);
        // the tensor-memory base as a RUN-TIME value (it is 0, checked above): with a compile-time base ptxas
        // folds the chained operand addresses of mma_f16_ts_tiles back into one constant + R2UR per MMA
        const uint32_t tmem_rt = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
        const uint64_t dXA = smem_desc_sw128(smem_u32(sXA));
        const uint64_t dW0 = smem_desc_sw128(smem_u32(sW));
        uint32_t s = 0, ph = 0, g = 0, m = 0, it = 0;
        auto next_stage = [&]() { if (++s == NSM) { s = 0; ph ^= 1; } };
        // SPLIT (single-thread issuer, 4-tile stages): the issuing thread's bookkeeping between two batches of MMAs
        // (a try_wait costs ~60 cycles even when the phase completed long ago) is not covered by queued MMAs -- the
        // layer-1 phase ran at ~44 cycles per MMA with all-zero operands too, i.e. not a power or data effect.  So
        // every wait is issued in the MIDDLE of a batch (after its first 8 MMAs): the W_FULL wait of the NEXT stage
        // and the hoisted accumulator hand-off; at a batch boundary only the commits remain.
        constexpr bool SPLIT = SINGLE && TPS == 4;
        // stages this CTA consumes in total (the W_FULL wait runs one stage ahead only while a next stage exists)
        const uint32_t total_stages = (uint32_t)(u1 - u0) * (uint32_t)(NC / G0 + NHID * NC * (KP / TPS));
        uint32_t q_stage = 0;
        uint32_t pre_n = 0;                 // upcoming ring stages whose W_FULL phase was already seen complete
        if (!SINGLE || elect_one()) {
        int cur_tile = -1;
        for (int u = u0; u < u1; ++u) {
            const int tile = CMBPO_TILE_OF(u);
            if (tile != cur_tile) {                 // a new row tile: its XA panel must have landed
                cur_tile = tile;
                mbar_wait(bar + X_FULL, it & 1);
                tc_fence_after();
                ++it;
            }
            {
                for (int j0 = 0; j0 < NC; j0 += G0) {       // layer 0: D = XA x W0 chunk (G0 chunks per stage)
                    if (pre_n) --pre_n; else mbar_wait(bar + W_FULL + s, ph);
                    ++q_stage;
#pragma unroll
                    for (int jj = 0; jj < G0; ++jj) {
                        // one chunk per instruction, buffer = chunk parity: the two epilogue pairs run as
                        // independent streams (one computes while the other is in its hand-off)
                        const uint32_t buf = g & 1, n = g >> 1;
                        mbar_wait(bar + D_EMPTY + buf, (n & 1) ^ 1);
                        tc_fence_after();
                        if (SINGLE || elect_one()) {
                            const uint64_t dB = dW0 + (uint64_t)((s * STAGE + jj * TILE) >> 4);
                            for (int ks = 0; ks < p.KS0; ++ks)
                                mma_f16(tmem + COL_D + buf * 64, dXA + 2 * ks, dB + 2 * ks, idesc_h, ks > 0);
                            mma_commit(bar + D_FULL + buf);
                            if (jj == G0 - 1) { if (CL == 2) mma_commit_mc(bar + W_EMPTY + s, 3); else mma_commit(bar + W_EMPTY + s); }
                        }
                        if (!SINGLE) __syncwarp();
                        g += 1;
                    }
                    next_stage();
                }
                for (int lyr = 0; lyr < NHID; ++lyr) {      // the HD x HD layers: middle ones (deep nets), then the last hidden
                const uint32_t col_a = (NMID > 0 && (lyr & 1)) ? COL_HB : COL_H1;     // A operand: the buffer the layer before wrote
                mbar_wait(bar + H1_FULL, (m * NHID + lyr) & 1);
                tc_fence_after();
                // layer 1.  The accumulator hand-off of chunk j+1 is waited for BEFORE the last stage of chunk j
                // is issued: the issue of that stage is back-pressured by the tensor pipe anyway, so the latency
                // of the (normally long satisfied) wait hides behind queued MMAs instead of opening a gap
                // between two chunks.
                {
                    const uint32_t buf0 = g & 1, n0 = g >> 1;
                    mbar_wait(bar + D_EMPTY + buf0, (n0 & 1) ^ 1);
                    tc_fence_after();
                }
                constexpr bool HOIST = (KP / TPS > 1);      // single-stage chunks (narrow members): wait per chunk
                for (int j = 0; j < NC; ++j) {
                    const uint32_t buf = g & 1;
                    if (!HOIST && j > 0) {
                        mbar_wait(bar + D_EMPTY + buf, ((g >> 1) & 1) ^ 1);
                        tc_fence_after();
                    }
                    for (int kq = 0; kq < KP / TPS; ++kq) {
                        if (pre_n) --pre_n; else mbar_wait(bar + W_FULL + s, ph);      // TMA completion: no tcgen05 fence needed
                        ++q_stage;
                        auto mid_waits = [&]() {
                            if (SPLIT && q_stage < total_stages) {       // the NEXT stage's weights
                                const uint32_t ns = (s + 1 == NSM) ? 0u : s + 1, nph = (s + 1 == NSM) ? (ph ^ 1u) : ph;
                                mbar_wait(bar + W_FULL + ns, nph);
                                pre_n = 1;
                            }
                            if (HOIST && kq == KP / TPS - 1 && j + 1 < NC) {
                                const uint32_t g1 = g + 1;
                                mbar_wait(bar + D_EMPTY + (g1 & 1), ((g1 >> 1) & 1) ^ 1);
                                tc_fence_after();
                            }
                        };
                        if (!SPLIT) mid_waits();
                        if (SINGLE || elect_one()) {
                            // TPS tiles x 4 K-steps from one asm statement (addresses chained inside, see tc_common.cuh)
                            if (SPLIT) {
                                const uint32_t a0 = tmem_rt + col_a + ((j / CPM) * KP + kq * TPS) * 32;
                                const uint64_t b0 = dW0 + (uint64_t)((s * STAGE) >> 4);
                                mma_f16_ts_tiles<2>(tmem + COL_D + buf * 64, a0, b0, idesc_h, kq > 0);
                                mid_waits();
                                mma_f16_ts_tiles<2>(tmem + COL_D + buf * 64, a0 + 64, b0 + (uint64_t)((2 * TILE) >> 4), idesc_h, 1u);
                            } else
                            mma_f16_ts_tiles<TPS>(tmem + COL_D + buf * 64, tmem_rt + col_a + ((j / CPM) * KP + kq * TPS) * 32,
                                                  dW0 + (uint64_t)((s * STAGE) >> 4), idesc_h, kq > 0);
                            if (CL == 2) mma_commit_mc(bar + W_EMPTY + s, 3); else mma_commit(bar + W_EMPTY + s);
                            if (kq == KP / TPS - 1) mma_commit(bar + D_FULL + buf);
                        }
                        if (!SINGLE) __syncwarp();
                        next_stage();
                    }
                    ++g;
                }
                }   // hidden-layer loop
                ++m;
            }
        }
        }
        __syncwarp();
    }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 112;");
        // ===== epilogue: 4 warpgroups; pair (wg>>1) owns accumulator buffer (wg>>1), half (wg&1) its columns =====
        const int wg = (warp - 4) >> 2;
        const uint32_t pair = (uint32_t)wg >> 1, half = (uint32_t)wg & 1;
        const int wq = hw_warp & 3;                // TMEM lane quarter this warp may access
        const int row = wq * 32 + lane;
        const uint32_t lane_base = (uint32_t)(wq * 32) << 16;
        const uint32_t bar_a = smem_u32(bar);
        uint32_t g = 0, m = 0, c1 = 0;
        // deferred OUT epilogue: the four warpgroups split the NP output columns (16 or 32 each)
        int prev_e = 0; long long prev_grow = 0; uint32_t prev_m = 0; bool have_prev = false;
        int prev_tile = 0;
        const int etid = (int)threadIdx.x - 128;                      // 0..511 among the epilogue threads
        // input scaler -> shared memory (identity when the net has none)
        if (etid < 64) {
            sIn[etid] = (p.mu_in && etid < p.K0) ? p.mu_in[etid] : 0.f;
            sIn[64 + etid] = (p.mu_in && etid < p.K0) ? p.sig_in[etid] : 1.f;
        }
        epi_bar();
        FzSmem fsm;
        if (FUSE) {
            fsm = fz_views(smem + SMEM_FZ);
            // small read-only vectors of the row math -> shared memory (no L1 in this carve-out: a global load per use
            // is an L2 round trip)
            const FusedStep& f = p.fz;
            for (int i = etid; i < f.c.D; i += 512) { fsm.sig[i] = f.c.sig_out[i]; fsm.mu[i] = f.c.mu_out[i]; fsm.l2s[i] = f.c.l2s_out[i]; }
            if (etid < f.A) fsm.log_std[etid] = f.log_std[etid];
            if (etid < f.n_elite && etid < 8) fsm.elite[etid] = f.c.elite[etid];
            epi_bar();
        }
        const int out_cw = (G > 1) ? p.NP : ((p.NP <= 64) ? 16 : 32);
        auto out_epilogue = [&]() {
            mbar_wait(bar + OUT_FULL, prev_m & 1);
            tc_fence_after();
            const int c_begin = wg * out_cw;
            uint32_t r[32];
            const bool mine = (G > 1) ? (wg < G && prev_e * G + wg < p.E) : (c_begin < p.NP);
            if (mine) {
                tmem_ld16(tmem + col_out + c_begin + lane_base, *reinterpret_cast<uint32_t(*)[16]>(&r[0]));
                if (out_cw == 32) tmem_ld16(tmem + col_out + c_begin + 16 + lane_base, *reinterpret_cast<uint32_t(*)[16]>(&r[16]));
                tmem_ld_wait();
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar + OUT_EMPTY);          // accumulator free again (16 warps arrive)
            if (FUSE) {
                // raw outputs -> tile-transposed L2 scratch (column-major inside the tile: a warp stores 32
                // consecutive floats per column), then the "last arriver" protocol: the CTA that delivers
                // the tile's E-th member runs the row math for the tile
                const FusedStep& f = p.fz;
                if (mine) {
                    const float* b2 = p.bias + (long long)prev_e * p.bias_stride + (1 + NHID) * HD;
                    float* dst = f.raw_tiles + ((size_t)prev_tile * p.E + prev_e) * p.Nout * 128 + row;
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        const int c = c_begin + i;
                        if (i < out_cw && c < p.Nout) __stcg(dst + (size_t)c * 128, __uint_as_float(r[i]) + __ldg(b2 + c));
                    }
                }
                __threadfence();
                epi_bar();
                if (etid == 0) {
                    const int old = atomicAdd(f.tile_cnt + prev_tile, 1);
                    const int last = (old == p.E - 1) ? 1 : 0;
                    if (last) f.tile_cnt[prev_tile] = 0;              // ready for the next step's launch
                    *fsm.flag = last;
                }
                epi_bar();
                if (*fsm.flag) {
                    __threadfence();
                    fused_rows(f, fsm, prev_tile, n_rows, etid);
                }
            } else
            if (mine && prev_grow < n_rows) {
                const int cb = (G > 1) ? 0 : c_begin;          // first output column of this warpgroup's slice
                float* orow = p.out + (long long)(prev_e * G + (G > 1 ? wg : 0)) * p.out_member_stride + prev_grow * p.Nout;
                const float* b2 = p.bias + (long long)prev_e * p.bias_stride + (1 + NHID) * HD + (G > 1 ? wg * p.NP : 0);
                if ((p.Nout & 3) == 0) {
#pragma unroll
                    for (int i = 0; i < 32; i += 4) {
                        const int c = cb + i;
                        if (i < out_cw && c < p.Nout) {
                            const float4 b = __ldg(reinterpret_cast<const float4*>(b2 + c));
                            float4 v;
                            v.x = __uint_as_float(r[i]) + b.x; v.y = __uint_as_float(r[i + 1]) + b.y;
                            v.z = __uint_as_float(r[i + 2]) + b.z; v.w = __uint_as_float(r[i + 3]) + b.w;
                            *reinterpret_cast<float4*>(orow + c) = v;
                        }
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        const int c = cb + i;
                        if (i < out_cw && c < p.Nout) orow[c] = __uint_as_float(r[i]) + b2[c];
                    }
                }
            }
            have_prev = false;
        };
        int cur_tile = -1;
        long long grow = 0;
        for (int u = u0; u < u1; ++u) {
            const int tile = CMBPO_TILE_OF(u);
            const bool new_tile = tile != cur_tile;
            cur_tile = tile;
            grow = (long long)tile * 128 + row;
            if (new_tile && wg == 0) {
                bool feed = grow < n_rows;
                const float* xr = p.x + grow * p.ldx;
                if (FUSE) {
                    // policy head of this row (what policy_rows_kernel does on the step-wise path): value heads,
                    // pending bootstraps, Gaussian head; the action goes to the per-row stash and, with the
                    // observation, into the XA panel below.  A tile shared by two CTAs is done by both: same
                    // inputs, same values.
                    const FusedStep& f = p.fz;
                    if (feed) {
                        const long long pth = f.row_path ? (long long)f.row_path[grow] : grow;
                        const float v = value_of(f.v, f.rules.B, grow), vc = value_of(f.vc, f.rules.B, grow);
                        const uint8_t pend = f.rules.pending[pth];
                        if (pend) {                                   // model_sampler.py:401-407 on s_{t+1}
                            if (pend & 1) f.rules.b.last_val[pth] = v;
                            if (pend & 2) f.rules.b.last_cval[pth] = vc;
                            f.rules.pending[pth] = 0;
                        }
                        feed = f.rules.alive[pth] != 0;
                        if (feed) {
                            f.vrow[grow] = v; f.vcrow[grow] = vc;
                            f.logp[grow] = policy_head_row<true>(f.pol_raw + grow * f.A, fsm.log_std,
                                                                 f.act_eps ? f.act_eps + pth * f.A : nullptr, f.seed,
                                                                 f.path_base + pth, f.rules.t, f.A, f.pi + grow * f.A,
                                                                 f.mu + grow * f.A);
                        }
                    }
                }
                // XA: this row of the input, scaled (pens/utils.py:156), 16-bit, zero padded to 64.  All global
                // loads of a 16-column batch are issued before the first use (one L2 round trip per 16 columns; the
                // earlier 8-column loop with the scaler vectors in global memory cost ~10 k cycles per row
                // tile with the MMA issuer waiting: shared memory is carved to the limit, there is no L1).
#pragma unroll 1
                for (int h = 0; h < 4; ++h) {
                    float v[16];
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i] = 0.f;
                    if (h * 16 < p.K0 + 2 * p.fold) {
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            const int k = h * 16 + i;
                            if (k < p.K0 && feed) {
                                if (FUSE) v[i] = (k < p.fz.O) ? p.fz.cur_obs[grow * p.fz.O + k] : p.fz.pi[grow * p.fz.A + (k - p.fz.O)];
                                else v[i] = xr[k];
                            }
                        }
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            const int k = h * 16 + i;
                            // fast division: the result is rounded to 16 bits right below (the IEEE
                            // version is a subroutine call inside this kernel)
                            if (k < p.K0 && feed) v[i] = __fdividef(__fsub_rn(v[i], sIn[k]), sIn[64 + k]);
                            else if (p.fold && feed && (k == p.K0 || k == p.K0 + 1)) v[i] = 1.0f;
                        }
                    }
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        uint4 q;
                        q.x = Cvt<FMT>::pack(v[8 * c], v[8 * c + 1]); q.y = Cvt<FMT>::pack(v[8 * c + 2], v[8 * c + 3]);
                        q.z = Cvt<FMT>::pack(v[8 * c + 4], v[8 * c + 5]); q.w = Cvt<FMT>::pack(v[8 * c + 6], v[8 * c + 7]);
                        *reinterpret_cast<uint4*>(sXA + panel_off(row, h * 2 + c)) = q;
                    }
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar + X_FULL);
            }
            {
                const int e = (int)(u % n_groups);
                // Each pair drains every other chunk (chunk j <-> accumulator buffer j&1 <-> pair), so the
                // loops below run over this pair's chunks only; they stay rolled (the fully unrolled variant
                // overflowed the instruction cache and doubled the drain time).  The unit's hidden biases
                // were copied to shared memory by the layer-2 producer warp.
                const float* sb = sBias + (m & 1) * (BIAS_SLOT / 4);
                mbar_wait_a(bar_a + 8 * (B_FULL + (m & 1)), (m >> 1) & 1);
                for (int i = 0; i < NC / 2; ++i) {               // layer-0 chunk j -> H1 columns
                    const int j = 2 * i + (int)pair;
                    const uint32_t gg = g + j, buf = pair, n = gg >> 1;
                    mbar_wait(bar + D_FULL + buf, n & 1);
                    tc_fence_after();
                    // WO, NMID = 1: H1 is the previous unit's layer-2 A operand (see the kernel comment)
                    const uint32_t h1_free = (WO && COL_LAST == COL_H1 && have_prev && i == 0) ? bar_a + 8 * OUT_FULL : 0u;
                    drain32<FMT, ACT>(tmem + COL_D + buf * 64 + half * 32 + lane_base, p.fold ? nullptr : sb + j * 64 + half * 32,
                                      tmem + COL_H1 + j * 32 + half * 16 + lane_base, bar_a + 8 * (D_EMPTY + buf),
                                      h1_free, WO ? (prev_m & 1) : 0u,
                                      ACT == 0 && p.member_act[e * G + j / CPM] != CMBPO_ACT_TANH);
                    __syncwarp();
                    if (lane == 0) mbar_arrive_a(bar_a + 8 * H1_FULL);
                }
                g += NC;
                // The previous member's OUT accumulator is drained HERE, after this member's layer-0
                // drains: the accumulator is not touched again before this member's first layer-2
                // MMA, so the global stores stay off the MMA warp's critical path.
                if (have_prev) out_epilogue();
                if (NMID > 0) {
                    for (int lyr = 1; lyr <= NMID; ++lyr) {      // middle layer lyr: chunk j -> the other hidden buffer
                        const uint32_t col_dst = (lyr & 1) ? COL_HB : COL_H1;
                        for (int i = 0; i < NC / 2; ++i) {
                            const int j = 2 * i + (int)pair;
                            const uint32_t gg = g + j, buf = pair, n = gg >> 1;
                            mbar_wait(bar + D_FULL + buf, n & 1);
                            tc_fence_after();
                            drain32<FMT, ACT>(tmem + COL_D + buf * 64 + half * 32 + lane_base, sb + lyr * HD + j * 64 + half * 32,
                                              tmem + col_dst + j * 32 + half * 16 + lane_base, bar_a + 8 * (D_EMPTY + buf), 0u, 0u);
                            __syncwarp();
                            if (lane == 0) mbar_arrive_a(bar_a + 8 * H1_FULL);
                        }
                        g += NC;
                    }
                }
                if constexpr (WO) {
                for (int i = 0; i < NC / 2; ++i) {               // last hidden layer, chunk j -> buffer LAST, K panel j
                    const int j = 2 * i + (int)pair;
                    const uint32_t gg = g + j, buf = pair, n = gg >> 1;
                    mbar_wait(bar + D_FULL + buf, n & 1);
                    tc_fence_after();
                    drain32<FMT, ACT>(tmem + COL_D + buf * 64 + half * 32 + lane_base, sb + NHID * HD + j * 64 + half * 32,
                                      tmem + COL_LAST + j * 32 + half * 16 + lane_base, bar_a + 8 * (D_EMPTY + buf), 0u, 0u);
                    __syncwarp();
                    if (lane == 0) mbar_arrive_a(bar_a + 8 * (HL_FULL + j));
                }
                } else
                for (int i = 0; i < NC / 2; ++i) {               // last hidden layer, chunk j -> an H2 buffer
                    const int j = 2 * i + (int)pair;
                    const uint32_t gg = g + j, buf = pair, n = gg >> 1, cc = c1 + j;
                    // H2 hand-off.  Double buffered: wait until the partial of chunk cc-2 (same buffer, same
                    // barrier, previous phase) has read it.  Single buffered: wait for the partial of chunk
                    // cc-1, which signals the OTHER pair's barrier (phase (cc-1)/2).  A single barrier shared
                    // by both pairs is wrong: a pair that is a whole phase ahead of the layer-2 issuer passes
                    // the parity test of the phase before (seen as an intermittent dead-lock with 256-wide
                    // nets and two-part outputs).
                    const uint32_t hbar = cc & 1, hn = cc >> 1, hb = (nh2 == 2) ? hbar : 0;
                    const uint32_t h2_free = (nh2 == 2) ? bar_a + 8 * (H2_EMPTY + hbar) : (cc == 0 ? 0u : bar_a + 8 * (H2_EMPTY + (hbar ^ 1)));
                    const uint32_t h2_par = (nh2 == 2) ? ((hn & 1) ^ 1) : ((((cc - 1) >> 1)) & 1);
                    mbar_wait(bar + D_FULL + buf, n & 1);
                    tc_fence_after();
                    drain32<FMT, ACT>(tmem + COL_D + buf * 64 + half * 32 + lane_base, sb + NHID * HD + j * 64 + half * 32,
                                      tmem + COL_H2 + hb * 32 + half * 16 + lane_base, bar_a + 8 * (D_EMPTY + buf),
                                      h2_free, h2_par, ACT == 0 && p.member_act[e * G + j / CPM] != CMBPO_ACT_TANH);
                    __syncwarp();
                    if (lane == 0) mbar_arrive_a(bar_a + 8 * (H2_FULL + hbar));
                }
                __syncwarp();
                if (lane == 0) mbar_arrive_a(bar_a + 8 * (B_EMPTY + (m & 1)));     // the bias buffer may be refilled
                g += NC; c1 += NC;
                prev_e = e; prev_grow = grow; prev_m = m; prev_tile = tile; have_prev = true;
                ++m;
            }
        }
        if (have_prev) out_epilogue();
    }
    tc_fence_before();
    __syncthreads();
    if (CL == 2) cluster_sync_all();      // the peer may still be signalling this CTA's barriers
#undef CMBPO_TILE_OF
    if (warp == 2) tmem_dealloc(tmem, 512);
}

// ---- weight packing -----------------------------------------------------------------------------
// W_l fp32 [E, K, M] (k-major rows, fc.py layout) -> stream of swizzled B tiles: tile row n = output
// neuron n0+n, 64 consecutive k from k0; zero padded.
//
// Two things are folded into the packed hidden layers (both exact in the 16-bit formats):
//  * swish members: W0, W1 (and the hidden biases) are HALVED, so the accumulators hold t = x/2 and the
//    epilogue evaluates swish(x) = t + t tanh t without the multiply;
//  * `fold`: the layer-0 bias rides in the GEMM -- rows K0 and K0+1 of the layer-0 tile hold the bias as a
//    (hi, lo) pair of 16-bit values (together ~21 mantissa bits) and the input panel holds 1.0 in those two
//    columns, which removes the bias add from the drain-bound layer-0 epilogue.  Needs K0 + 2 <= 64.
struct PackCfg { int fold; int act[CMBPO_MAX_E]; };
struct PackW { const float* W[CMBPO_MAX_LAYERS]; int n_layers; };     // fp32 master copies, W[n_layers-1] = output layer

template <int FMT> __device__ __forceinline__ uint16_t to16(float v) {
    if (FMT == 0) { __half x = __float2half_rn(fminf(fmaxf(v, -65504.f), 65504.f)); return *reinterpret_cast<uint16_t*>(&x); }
    __nv_bfloat16 x = __float2bfloat16_rn(v); return *reinterpret_cast<uint16_t*>(&x);
}
template <int FMT> __device__ __forceinline__ float from16(uint16_t h) {
    if (FMT == 0) return __half2float(*reinterpret_cast<__half*>(&h));
    return __bfloat162float(*reinterpret_cast<__nv_bfloat16*>(&h));
}

template <int FMT>
__global__ void pack_weights_kernel(PackW pw, const float* b0, int K0, int HD,
                                    int Nout, int E, int group, const Stage* stages, int n_stages,
                                    unsigned long long member_bytes, PackCfg cfg, uint8_t* out) {
    // HD = the REAL hidden width of the fp32 master copy; tiles beyond it (the instantiation's padded width) are zeros
    const Stage st = stages[blockIdx.x];
    const int e = blockIdx.y * group + st.member;        // real member (may be >= E in the last group: zeros)
    const float* W; int K, M;
    const int last = pw.n_layers - 1;                    // st.layer indexes the master copies
    if (st.layer == 0) { W = pw.W[0] + (size_t)e * K0 * HD; K = K0; M = HD; }
    else if (st.layer < last) { W = pw.W[st.layer] + (size_t)e * HD * HD; K = HD; M = HD; }
    else { W = pw.W[last] + (size_t)e * HD * Nout; K = HD; M = Nout; }
    if (e >= E) K = 0;
    const float scale = (st.layer < last && e < E && cfg.act[e] == CMBPO_ACT_SWISH) ? 0.5f : 1.0f;
    uint8_t* dst = out + (size_t)blockIdx.y * member_bytes + st.off;
    for (int idx = threadIdx.x; idx < st.rows * 64; idx += blockDim.x) {
        const int n = idx >> 6, k = idx & 63;
        const int gk = st.k0 + k, gn = st.n0 + n;
        float v = (gk < K && gn < M) ? scale * W[(size_t)gk * M + gn] : 0.f;
        uint16_t h = to16<FMT>(v);
        if (st.layer == 0 && cfg.fold && e < E && gn < M && (gk == K0 || gk == K0 + 1)) {
            const float b = scale * b0[(size_t)e * HD + gn];
            const uint16_t hi = to16<FMT>(b);
            h = (gk == K0) ? hi : to16<FMT>(b - from16<FMT>(hi));
        }
        *reinterpret_cast<uint16_t*>(dst + panel_off(n, k >> 3) + (k & 7) * 2) = h;
    }
}

// per unit: [b_0 of the G members | ... | b_{nh-1} of the G members | b_out (NP each) of the G members]; HD = padded
// member width (layout), HR = real width of the master copy, nh = number of hidden layers.  The hidden biases of
// swish members are halved like their weights.
struct PackB { const float* b[CMBPO_MAX_LAYERS]; int nh; };
__global__ void pack_bias_kernel(PackB pb, int HD, int HR, int Nout, int NP, int E, int group, PackCfg cfg, float* out) {
    const int u = blockIdx.x;
    const int stride = group * (pb.nh * HD + NP);
    for (int i = threadIdx.x; i < stride; i += blockDim.x) {
        float v = 0.f;
        if (i < pb.nh * group * HD) {
            const int l = i / (group * HD), k = i - l * group * HD, e = u * group + k / HD;
            if (e < E && k % HD < HR) v = pb.b[l][(size_t)e * HR + k % HD] * (cfg.act[e] == CMBPO_ACT_SWISH ? 0.5f : 1.0f);
        } else {
            const int k = i - pb.nh * group * HD, e = u * group + k / NP, c = k % NP;
            if (e < E && c < Nout) v = pb.b[pb.nh][(size_t)e * Nout + c];
        }
        out[(size_t)u * stride + i] = v;
    }
}

// hidden width padded to a kernel instantiation (zero weights / biases: swish(0) = tanh(0) = 0, so the padded neurons
// contribute nothing to the next layer)
int padded_hd(int h) { return h <= 128 ? 128 : (h <= 256 ? 256 : 512); }

struct OutShape { int NP, parts; };
OutShape out_shape(int Nout) {
    if (Nout <= 64) return {((Nout + 15) / 16) * 16, 1};
    return {((Nout + 31) / 32) * 32, 2};       // two N-halves, each a multiple of 16
}

// the order in which the MMA warp consumes weight tiles (must match the kernel's loops):
// main stream = layer-0 chunk tiles, then per chunk the layer-1 K-panel tiles; W2 stream = per chunk
// the layer-2 tile(s).  The wide-output deep kernels (WO) read a two-part chunk as ONE tile of NP rows: tile
// rows are 128 B apart and NP/2 is a multiple of 8, so the q = 1 tile starts exactly at row NP/2 of it.
void stage_programs(int HD, int NP, int parts, int group, int nhid, std::vector<Stage>* main_prog,
                    unsigned long long* main_bytes, std::vector<Stage>* w2_prog, unsigned long long* w2_bytes) {
    // nhid = number of HD x HD layers (1 + NMID); Stage.layer indexes the master copies: 0, 1 .. nhid, nhid + 1 = output
    // HD = virtual width of a unit (group * member width); chunk j belongs to member j / CPM
    const int NC = HD / 64, CPM = NC / group, KPm = HD / 64 / group, NPp = NP / parts;
    unsigned long long off = 0;
    for (int j = 0; j < NC; ++j) { main_prog->push_back(Stage{0, (j % CPM) * 64, 0, 64, j / CPM, off}); off += TILE; }
    for (int lyr = 1; lyr <= nhid; ++lyr)
        for (int j = 0; j < NC; ++j)
            for (int kp = 0; kp < KPm; ++kp) {
                main_prog->push_back(Stage{lyr, (j % CPM) * 64, kp * 64, 64, j / CPM, off});
                off += TILE;
            }
    *main_bytes = off;
    off = 0;
    for (int j = 0; j < NC; ++j)
        for (int q = 0; q < parts; ++q) {
            w2_prog->push_back(Stage{nhid + 1, q * NPp, (j % CPM) * 64, NPp, j / CPM, off});
            off += (unsigned long long)NPp * 128;
        }
    *w2_bytes = off;
}

int chunks_per_w2_slot(int HD, int NP, int slot_bytes = W2SLOT) {
    int cps = slot_bytes / (NP * 128);
    int p2 = 1;
    while (p2 * 2 <= cps) p2 *= 2;
    const int NC = HD / 64;
    return p2 < NC ? p2 : NC;
}

template <int HD, int FMT, int ACT, int G = 1, bool FUSE = false, int NMID = 0, bool WO = false>
int launch_tc(cmbpo_ctx* ctx, const TcParams& p) {
    const int smem = (FUSE ? SMEM_TOTAL_F : SMEM_TOTAL) + 1024;
    static_assert(SMEM_TOTAL + 1024 <= 232448, "shared memory budget");
    auto kern = ens_mlp3_tc_kernel<HD, FMT, ACT, G, FUSE, NMID, 1, WO>;
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const long long units = (long long)p.ntiles * ((p.E + G - 1) / G);
    const int grid = units < ctx->sm_count ? (int)units : ctx->sm_count;
    kern<<<grid, NTHREADS, smem, ctx->stream>>>(p);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// cluster pairs (CL = 2, see the kernel): wide ordinary ensembles with enough row tiles.  The number of co-resident
// pairs is asked of the runtime once per kernel (a GPC with an odd SM count leaves one SM without a partner).
template <int HD, int FMT, int ACT>
int launch_tc_pairs(cmbpo_ctx* ctx, const TcParams& p) {
    const int smem = SMEM_TOTAL + 1024;
    auto kern = ens_mlp3_tc_kernel<HD, FMT, ACT, 1, false, 0, 2>;
    static int max_pairs = -1;
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.blockDim = dim3(NTHREADS); cfg.dynamicSmemBytes = smem; cfg.stream = ctx->stream;
    cfg.attrs = attr; cfg.numAttrs = 1;
    if (max_pairs < 0) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        cfg.gridDim = dim3(2 * (ctx->sm_count / 2));
        int n = 0;
        if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) {      // no cluster support here: ordinary launch
            (void)cudaGetLastError();
            n = 0;
        }
        max_pairs = n < 1 ? 0 : (n > ctx->sm_count / 2 ? ctx->sm_count / 2 : n);
        // pairs are worth ~2 %; a part whose GPC layout leaves more than two SMs without a partner loses more than that
        if (2 * max_pairs < ctx->sm_count - 2) max_pairs = 0;
    }
    if (max_pairs == 0) return launch_tc<HD, FMT, ACT>(ctx, p);
    const long long units = (long long)((p.ntiles + 1) / 2) * p.E;
    const int pairs = units < max_pairs ? (int)units : max_pairs;
    cfg.gridDim = dim3(2 * pairs);
    CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, p));
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// the fused rollout step: swish dynamics ensembles of any supported width
template <int FMT>
int launch_tc_fused(cmbpo_ctx* ctx, const TcParams& p, int hd) {
    if (hd == 128) return launch_tc<128, FMT, CMBPO_ACT_SWISH, 1, true>(ctx, p);
    if (hd == 256) return launch_tc<256, FMT, CMBPO_ACT_SWISH, 1, true>(ctx, p);
    return launch_tc<512, FMT, CMBPO_ACT_SWISH, 1, true>(ctx, p);
}

template <int HD, int FMT>
int launch_tc_act(cmbpo_ctx* ctx, const TcParams& p, int act) {
    if (act == 0) return launch_tc<HD, FMT, 0>(ctx, p);
    if (act == CMBPO_ACT_SWISH) return launch_tc<HD, FMT, CMBPO_ACT_SWISH>(ctx, p);
    return launch_tc<HD, FMT, CMBPO_ACT_TANH>(ctx, p);
}

// 3 / 4 hidden layers at (padded) width 256; more than 64 output columns take the wide-output kernel (WO)
template <int FMT, int ACT, int NMID>
int launch_tc_deep_out(cmbpo_ctx* ctx, const TcParams& p) {
    if (p.NP > 64) return launch_tc<256, FMT, ACT, 1, false, NMID, true>(ctx, p);
    return launch_tc<256, FMT, ACT, 1, false, NMID>(ctx, p);
}
template <int FMT>
int launch_tc_deep(cmbpo_ctx* ctx, const TcParams& p, int act, int nmid) {
    if (act == CMBPO_ACT_SWISH)
        return nmid == 1 ? launch_tc_deep_out<FMT, CMBPO_ACT_SWISH, 1>(ctx, p)
                         : launch_tc_deep_out<FMT, CMBPO_ACT_SWISH, 2>(ctx, p);
    return nmid == 1 ? launch_tc_deep_out<FMT, CMBPO_ACT_TANH, 1>(ctx, p)
                     : launch_tc_deep_out<FMT, CMBPO_ACT_TANH, 2>(ctx, p);
}

template <int FMT>
int launch_tc_grouped(cmbpo_ctx* ctx, const TcParams& p, int act) {       // 4 members of width 128 per unit
    if (act == 0) return launch_tc<512, FMT, 0, 4>(ctx, p);
    if (act == CMBPO_ACT_SWISH) return launch_tc<512, FMT, CMBPO_ACT_SWISH, 4>(ctx, p);
    return launch_tc<512, FMT, CMBPO_ACT_TANH, 4>(ctx, p);
}

template <int FMT>
int launch_tc_hd(cmbpo_ctx* ctx, const TcParams& p, int hd, int act) {
    if (hd == 128) return launch_tc_act<128, FMT>(ctx, p, act);
    if (hd == 256) return launch_tc_act<256, FMT>(ctx, p, act);
    if (p.ntiles >= 2) {
        if (act == CMBPO_ACT_SWISH) return launch_tc_pairs<512, FMT, CMBPO_ACT_SWISH>(ctx, p);
        return launch_tc_pairs<512, FMT, CMBPO_ACT_TANH>(ctx, p);
    }
    if (act == CMBPO_ACT_SWISH) return launch_tc<512, FMT, CMBPO_ACT_SWISH>(ctx, p);
    return launch_tc<512, FMT, CMBPO_ACT_TANH>(ctx, p);
}

}  // namespace

// 2 hidden layers: any equal width <= 512 (padded to 128 / 256 / 512), <= 64 inputs, <= 128 outputs; <= 96 outputs
// above width 256 (tensor memory: at width 512 the OUT accumulator of a 128-column output, 512 - NP = column 384,
// would overlap the single H2 buffer at columns 384-415).
// 3 or 4 hidden layers (e.g. the (200,200,200,200) default of algorithms/cmbpo.py:54): equal width <= 256, <= 64
// inputs, <= 128 outputs (tensor memory: two hidden buffers, the accumulators and OUT fill the 512 columns; above 64
// outputs the last hidden layer's buffer is layer 2's A operand, see WO at the kernel).
bool ens_tc_supported(const Net& n) {
    if (!n.loaded || n.n_layers < 3 || n.n_layers > 5) return false;
    const int hd = n.dims[1], L = n.n_layers;
    for (int l = 1; l < L; ++l) if (n.dims[l] != hd) return false;
    if (hd < 1 || hd > (L == 3 ? 512 : 256)) return false;
    if (n.dims[0] > 64 || n.dims[L] > ((L == 3 && hd > 256) ? 96 : 128)) return false;
    for (int l = 1; l < L - 1; ++l) if (n.acts[l] != n.acts[0]) return false;
    if (n.acts[L - 1] != CMBPO_ACT_NONE) return false;
    return n.acts[0] == CMBPO_ACT_SWISH || n.acts[0] == CMBPO_ACT_TANH;
}

// pack both 16-bit formats once per weight upload: [main stream | W2 stream] per precision
int ens_tc_prepare(cmbpo_ctx* ctx, Net& net) {
    const int L = net.n_layers, nhid = L - 2;            // HD x HD layers
    const int HR = net.dims[1], HD = (nhid > 1) ? 256 : padded_hd(HR), K0 = net.dims[0], Nout = net.dims[L];
    net.tc_hd = HD;
    const OutShape os = out_shape(Nout);
    // narrow ensembles run grouped: 4 members of width 128 per unit (their OUT blocks share 64 columns)
    const int group = (nhid == 1 && HD == 128 && net.E >= 2 && os.NP <= 16) ? 4 : 1;
    const int n_units = (net.E + group - 1) / group;
    net.tc_group = group;
    unsigned long long main_bytes = 0, w2_bytes = 0;
    std::vector<Stage> mp, wp;
    stage_programs(HD * group, os.NP, os.parts, group, nhid, &mp, &main_bytes, &wp, &w2_bytes);
    PackW pw; PackB pb;
    pw.n_layers = L; pb.nh = L - 1;
    for (int l = 0; l < CMBPO_MAX_LAYERS; ++l) { pw.W[l] = net.W[l]; pb.b[l] = net.b[l]; }
    PackCfg pc;
    pc.fold = (K0 + 2 <= 64) ? 1 : 0;
    for (int e = 0; e < CMBPO_MAX_E; ++e) pc.act[e] = net.member_act[0] >= 0 ? net.member_act[e] : net.acts[0];
    net.tc_fold = pc.fold;
    Stage *d_mp, *d_wp;
    CUDA_TRY(cudaMalloc(&d_mp, mp.size() * sizeof(Stage)));
    CUDA_TRY(cudaMalloc(&d_wp, wp.size() * sizeof(Stage)));
    CUDA_TRY(cudaMemcpyAsync(d_mp, mp.data(), mp.size() * sizeof(Stage), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(d_wp, wp.data(), wp.size() * sizeof(Stage), cudaMemcpyHostToDevice, ctx->stream));
    for (int prec = CMBPO_PREC_BF16; prec <= CMBPO_PREC_FP16; ++prec) {
        const size_t total = (size_t)n_units * (main_bytes + w2_bytes);
        CUDA_TRY(cudaMalloc(&net.tc_pack[prec], total));
        net.tc_pack_bytes[prec] = (size_t)main_bytes;       // W2 stream starts at E * main_bytes
        uint8_t* base = (uint8_t*)net.tc_pack[prec];
        uint8_t* base2 = base + (size_t)n_units * main_bytes;
        dim3 g1((unsigned)mp.size(), n_units), g2((unsigned)wp.size(), n_units);
        if (prec == CMBPO_PREC_FP16) {
            pack_weights_kernel<0><<<g1, 256, 0, ctx->stream>>>(pw, net.b[0], K0, HR, Nout, net.E, group, d_mp, (int)mp.size(), main_bytes, pc, base);
            pack_weights_kernel<0><<<g2, 256, 0, ctx->stream>>>(pw, net.b[0], K0, HR, Nout, net.E, group, d_wp, (int)wp.size(), w2_bytes, pc, base2);
        } else {
            pack_weights_kernel<1><<<g1, 256, 0, ctx->stream>>>(pw, net.b[0], K0, HR, Nout, net.E, group, d_mp, (int)mp.size(), main_bytes, pc, base);
            pack_weights_kernel<1><<<g2, 256, 0, ctx->stream>>>(pw, net.b[0], K0, HR, Nout, net.E, group, d_wp, (int)wp.size(), w2_bytes, pc, base2);
        }
    }
    CUDA_TRY(cudaMalloc(&net.tc_bias, (size_t)n_units * group * ((L - 1) * HD + os.NP) * sizeof(float)));
    pack_bias_kernel<<<n_units, 256, 0, ctx->stream>>>(pb, HD, HR, Nout, os.NP, net.E, group, pc, net.tc_bias);
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    CUDA_TRY(cudaFree(d_mp));
    CUDA_TRY(cudaFree(d_wp));
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// the conditions under which cmbpo_rollout may fuse the step around this ensemble's GEMM chain
bool ens_tc_fusable(const Net& n) {
    if (!ens_tc_supported(n) || n.n_layers != 3 || n.tc_group != 1 || n.E != 7 || !n.probabilistic) return false;
    if (n.acts[0] != CMBPO_ACT_SWISH || n.member_act[0] >= 0) return false;
    const OutShape os = out_shape(n.dims[3]);
    return os.NP * 128 <= W2SLOT_F && n.D <= 64;       // one chunk's layer-2 tiles must fit a (shrunk) ring slot
}

int ens_tc_fused_rp_shift(int O) {
    // rows per row-math pass: kl + epv staging of [O][RP] floats each within FZ_STAGE
    int sh = 7;
    while (sh > 5 && (size_t)(1 << sh) * O * 8 > (size_t)FZ_STAGE) --sh;
    return ((size_t)(1 << sh) * O * 8 <= (size_t)FZ_STAGE) ? sh : -1;
}

int ens_forward_tc(cmbpo_ctx* ctx, Net& net, const float* x, int64_t N, float* out_raw, int precision,
                   const int64_t* n_dev, const FusedStep* fz) {
    CMBPO_CHECK(precision == CMBPO_PREC_BF16 || precision == CMBPO_PREC_FP16, "bad precision %d", precision);
    CMBPO_CHECK(net.tc_pack[precision], "tcgen05 weights not packed");
    if (N <= 0) return 0;
    CMBPO_CHECK((N + 127) / 128 * (int64_t)net.E < (int64_t)1 << 31, "too many rows for one launch");
    const int HD = net.tc_hd;                   // padded hidden width = kernel instantiation
    const int nmid = net.n_layers - 3;          // middle hidden layers (deep variant)
    const OutShape os = out_shape(net.dims[net.n_layers]);
    TcParams p;
    p.Nout = net.dims[net.n_layers];
    p.NP = os.NP; p.parts = os.parts;
    p.cps = chunks_per_w2_slot(HD * net.tc_group, os.NP, fz ? W2SLOT_F : W2SLOT);
    p.wmain = (const uint8_t*)net.tc_pack[precision];
    p.main_bytes = net.tc_pack_bytes[precision];
    p.w2 = p.wmain + (size_t)((net.E + net.tc_group - 1) / net.tc_group) * p.main_bytes;
    p.w2_bytes = (unsigned long long)(HD * net.tc_group / 64) * p.NP * 128;
    const int group = net.tc_group;
    p.bias = net.tc_bias; p.bias_stride = group * ((net.n_layers - 1) * HD + p.NP);
    p.E = net.E; p.K0 = net.dims[0]; p.fold = net.tc_fold; p.KS0 = (p.K0 + (p.fold ? 2 : 0) + 15) / 16;
    p.x = x; p.N = N; p.ldx = net.dims[0];
    p.n_dev = reinterpret_cast<const long long*>(n_dev);
    p.mu_in = net.has_in ? net.mu_in : nullptr; p.sig_in = net.sig_in;
    p.out = out_raw; p.out_member_stride = (long long)N * p.Nout;
    p.ntiles = (int)((N + 127) / 128);
    for (int i = 0; i < CMBPO_MAX_E; ++i) p.member_act[i] = net.member_act[i];
    if (fz) {
        CMBPO_CHECK(ens_tc_fusable(net) && fz->rp_shift >= 5, "this ensemble cannot run the fused rollout step");
        p.fz = *fz;
        return precision == CMBPO_PREC_FP16 ? launch_tc_fused<0>(ctx, p, HD) : launch_tc_fused<1>(ctx, p, HD);
    }
    memset(&p.fz, 0, sizeof(p.fz));
    const int act_sel = net.member_act[0] >= 0 ? 0 : net.acts[0];
    if (nmid > 0) {
        CMBPO_CHECK(HD == 256 && group == 1 && (nmid == 1 || nmid == 2) && net.member_act[0] < 0, "deep tcgen05 variant: bad shape");
        return precision == CMBPO_PREC_FP16 ? launch_tc_deep<0>(ctx, p, act_sel, nmid) : launch_tc_deep<1>(ctx, p, act_sel, nmid);
    }
    if (group == 4) return precision == CMBPO_PREC_FP16 ? launch_tc_grouped<0>(ctx, p, act_sel) : launch_tc_grouped<1>(ctx, p, act_sel);
    if (precision == CMBPO_PREC_FP16) return launch_tc_hd<0>(ctx, p, HD, act_sel);
    return launch_tc_hd<1>(ctx, p, HD, act_sel);
}
