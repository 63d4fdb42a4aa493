// Shared declarations of libcmbpo_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/cmbpo_b200.h"

#define CMBPO_MAX_LAYERS 8
#define CMBPO_MAX_E 8        // members held in registers by the per-row math
#define CMBPO_MAX_OBS 64     // per-row register arrays
#define CMBPO_MAX_ACT 32

void cmbpo_set_error(const char* fmt, ...);

#define CUDA_TRY(expr)                                                                   \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess) {                                                         \
            cmbpo_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                            __LINE__);                                                   \
            return 1;                                                                    \
        }                                                                                \
    } while (0)

#define CMBPO_CHECK(cond, ...)           \
    do {                                 \
        if (!(cond)) {                   \
            cmbpo_set_error(__VA_ARGS__); \
            return 1;                    \
        }                                \
    } while (0)

// One MLP ensemble resident in HBM.  fp32 master copy in the reference's layout
// (fc.py:135-139: W [E,in,out], b [E,out]) + pre-packed 16-bit tiles for the tcgen05 path.
struct Net {
    bool loaded = false;
    int E = 0, n_layers = 0;
    int dims[CMBPO_MAX_LAYERS + 1] = {0};
    int acts[CMBPO_MAX_LAYERS] = {0};
    float* W[CMBPO_MAX_LAYERS] = {nullptr};
    float* b[CMBPO_MAX_LAYERS] = {nullptr};
    bool probabilistic = false;
    int D = 0;                  // output width seen by callers (half the last layer if probabilistic)
    bool has_in = false, has_out = false;
    float *mu_in = nullptr, *sig_in = nullptr;                       // [in]; sigma = max(sqrt(var),1e-2)
    float *mu_out = nullptr, *sig_out = nullptr, *l2s_out = nullptr; // [D]; l2s = 2*log(sigma)
    int n_elite = 0;
    int* elite = nullptr;       // device [n_elite]
    // tcgen05 path: weights packed as ready-to-copy shared-memory tile images (see ens_tc.cu)
    void* tc_pack[3] = {nullptr, nullptr, nullptr};   // per precision (index = CMBPO_PREC_*)
    size_t tc_pack_bytes[3] = {0, 0, 0};
    float* tc_bias = nullptr;   // biases re-laid for the epilogue
    int tc_group = 1;           // members per tcgen05 work unit (4 for narrow ensembles)
    int tc_hd = 0;              // hidden width padded to the kernel instantiation (128 / 256 / 512)
    int tc_fold = 0;            // layer-0 bias folded into the packed layer-0 tiles (input dim + 2 <= 64)
    // merged nets only: hidden activation per member (CMBPO_ACT_*); all -1 for an ordinary ensemble
    int member_act[CMBPO_MAX_E] = {-1, -1, -1, -1, -1, -1, -1, -1};
};

struct Workspace {
    void* ptr = nullptr;
    size_t bytes = 0;
};

struct ProfSlot {
    std::vector<cudaEvent_t> start, stop;
    size_t used = 0;
};

struct cmbpo_ctx {
    bool profile = false;
    ProfSlot prof[CMBPO_PROF_SLOTS];
    int device = 0;
    cudaStream_t stream = nullptr;
    int sm_count = 148;
    Net nets[CMBPO_NET_COUNT];
    // actor + V + VC merged into ONE ensemble sharing one input panel (tcgen05 path only): member 0 =
    // actor, then the V members, then the VC members; each member's own input scaler is folded into
    // its first layer relative to the common transform (policy_pack.cu)
    Net polnet;
    int pol_nv = 0, pol_nvc = 0;
    float* log_std = nullptr;   // [A]
    int A = 0;
    Workspace ws[8];            // reusable scratch slots
    int64_t launches = 0;
    // per-context (= per-device) records of cudaFuncSetAttribute calls already made
    size_t step_smem_max[2] = {0, 0};
    bool gae_rows_attr_set = false;
    // rollout: page-locked mirror of the live row count + events (early exit once every path ended)
    int64_t* host_n = nullptr;      // [4]
    cudaEvent_t n_ev[4] = {nullptr, nullptr, nullptr, nullptr};
    // ensemble training (train.cu): optimiser state, activations and the cuBLAS handle per network slot
    void* train[CMBPO_NET_COUNT] = {nullptr};
};

// grow-only scratch
int cmbpo_ws_get(cmbpo_ctx* ctx, int slot, size_t bytes, void** out);

// RAII bracket: records start/stop events around a launch when profiling is on
struct ProfScope {
    cmbpo_ctx* ctx; int slot; bool on;
    ProfScope(cmbpo_ctx* c, int s) : ctx(c), slot(s), on(c->profile && s >= 0) {
        if (!on) return;
        ProfSlot& p = ctx->prof[slot];
        if (p.used == p.start.size()) {
            cudaEvent_t a, b;
            cudaEventCreate(&a); cudaEventCreate(&b);
            p.start.push_back(a); p.stop.push_back(b);
        }
        cudaEventRecord(p.start[p.used], ctx->stream);
    }
    ~ProfScope() {
        if (!on) return;
        ProfSlot& p = ctx->prof[slot];
        cudaEventRecord(p.stop[p.used], ctx->stream);
        p.used++;
    }
};

static inline int cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// ---- internal entry points shared between translation units -------------------------------
// fp32 CUDA-core MLP chain: X [N,in] (or [E,N,in]) -> raw last-layer output [E,N,dims[L]]
int ens_forward_f32(cmbpo_ctx* ctx, const Net& net, const float* x, int64_t N, bool x_is_3d,
                    float* out_raw);
// tcgen05 MLP chain (2 hidden layers), same contract
struct FusedStep;       // step_common.cuh
int ens_forward_tc(cmbpo_ctx* ctx, Net& net, const float* x, int64_t N, float* out_raw,
                   int precision, const int64_t* n_dev = nullptr, const FusedStep* fz = nullptr);
bool ens_tc_fusable(const Net& net);
int ens_tc_fused_rp_shift(int obs_dim);
bool ens_tc_supported(const Net& net);
int ens_tc_prepare(cmbpo_ctx* ctx, Net& net);
int policy_pack_build(cmbpo_ctx* ctx);
void net_free(Net& n);
void train_free(cmbpo_ctx* ctx, int which);
// n_dev (tcgen05 precisions only): live row count in device memory, <= N; rows beyond it are skipped
int ens_forward(cmbpo_ctx* ctx, Net& net, const float* x, int64_t N, bool x_is_3d, float* out_raw,
                int precision, const int64_t* n_dev = nullptr);
