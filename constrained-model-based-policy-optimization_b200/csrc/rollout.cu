// Step-wise model rollout (policy -> dynamics ensemble -> FakeEnv row math -> sampler rules ->
// ModelBuffer write-out) and the single-step entry points cmbpo_policy_act / cmbpo_fakeenv_step.
//
// The GEMM chains go through ens_forward(precision): fp32 CUDA cores (logic reference on the
// device) or the tcgen05 kernels of ens_tc.cu.  The per-row arithmetic lives in row_math.cuh.
//
// Reference: samplers/model_sampler.py:239-375 (sample), 377-416 (_finish_paths),
//            models/fake_env.py:66-172, buffers/modelbuffer.py:114-135 (store_multiple),
//            policies/cpo_policy.py:801-835.
#include <cstdlib>
#include <cstring>
#include "common.cuh"
#include "row_math.cuh"

namespace {

// one non-probabilistic value ensemble read through PE.predict (cpo_policy.py:801-835, pe.py:343)
struct ValueHead {
    const float* raw;         // [E, N, ld], value in column 0
    int E, ld;
    const float *mu_out, *sig_out;   // [1] or null
};

__device__ __forceinline__ float value_of(const ValueHead& h, int64_t N, int64_t p) {
    // tf.reduce_mean over members of inverse_transform(out) (pe.py:343, pens/utils.py:167)
    float s = 0.f;
    for (int e = 0; e < h.E; ++e) {
        float m = h.raw[((int64_t)e * N + p) * h.ld];
        if (h.mu_out) m = __fadd_rn(__fmul_rn(h.sig_out[0], m), h.mu_out[0]);
        s = (e == 0) ? m : __fadd_rn(s, m);
    }
    return __fdiv_rn(s, (float)h.E);
}

struct PolicyRowsArgs {
    int64_t N;                 // rows
    int O, A;
    const float* obs;          // [N,O]
    const float* mu_raw;       // [N,A] actor output
    const float* log_std;      // [A]
    ValueHead v, vc;
    const float* eps;          // [N,A] or null
    const int32_t* path_ids;   // [N] or null
    int64_t path_base;
    uint64_t seed;
    int step;
    const uint8_t* alive;      // [paths] or null (all rows)
    const int32_t* row_path;   // [N] compact row -> local path index, or null (row == path)
    const int64_t* n_dev;      // live row count on the device (<= N), or null (all N rows)
    // outputs
    float *pi, *logp, *mu, *vout, *vcout;   // [N,A],[N],[N,A],[N],[N]; any may be null
    float* xin;                // [N, O+A] concat(obs, pi) or null
    // pending bootstraps (rollout only)
    uint8_t* pending;          // [N] bit0: last_val, bit1: last_cval
    float *last_val, *last_cval;
};

constexpr int POLICY_ROWS = 128;      // rows per block of policy_rows_kernel
constexpr int POLICY_THREADS = 384;   // 128 row threads + 256 threads for the (row, four action dims) items

// Phase 1 runs two kinds of threads side by side (a row's work done by ONE thread is a ~50 k-cycle dependent
// chain -- value-head loads, a Philox block and two Box-Muller pairs per four action dims, exp / divide per dim --
// and 100 k rows are only ~5 warps per scheduler, so that version was bound by its own latency: 27 us per launch):
//   threads [0,128)    one per row: value heads, pending bootstraps (model_sampler.py:401-407)
//   threads [128,384)  one per (row, quad of action dims): the Gaussian head's noise, pi and log-density
//                      terms of those dims (ac_network.py:105-111, 46-48), pi / mu written out
// then the row thread adds the row's terms in numpy's order (the same additions in the same order as before:
// bit-identical).  Phase 2, all threads: the block's [128, O+A] slice of the dynamics input `xin` = concat(obs, pi)
// is one contiguous range -> written with consecutive threads on consecutive floats.
template <bool FAST>
__global__ void __launch_bounds__(POLICY_THREADS) policy_rows_kernel(PolicyRowsArgs a) {
    __shared__ float s_pi[POLICY_ROWS * CMBPO_MAX_ACT];
    __shared__ float s_term[POLICY_ROWS * CMBPO_MAX_ACT];
    __shared__ unsigned char s_live[POLICY_ROWS];
    const int64_t base = (int64_t)blockIdx.x * POLICY_ROWS;
    const int64_t n_rows = a.n_dev ? *a.n_dev : a.N;
    const int A = a.A;
    if (threadIdx.x < POLICY_ROWS) {
        const int64_t r = base + threadIdx.x;          // row of the (possibly compacted) batch
        bool live = r < n_rows;
        if (live) {
            const int64_t p = a.row_path ? (int64_t)a.row_path[r] : r;   // path the per-path arrays are indexed by
            const float v = value_of(a.v, a.N, r), vc = value_of(a.vc, a.N, r);
            if (a.pending) {
                uint8_t f = a.pending[p];
                if (f) {                                   // model_sampler.py:401-407 on s_{t+1}
                    if (f & 1) a.last_val[p] = v;
                    if (f & 2) a.last_cval[p] = vc;
                    a.pending[p] = 0;
                }
            }
            live = !(a.alive && !a.alive[p]);
            if (live) {
                if (a.vout) a.vout[r] = v;
                if (a.vcout) a.vcout[r] = vc;
            }
            live = live && a.mu_raw;
        }
        s_live[threadIdx.x] = live ? 1 : 0;
    } else if (a.mu_raw) {
        const int NQ = (A + 3) >> 2;
        for (int it = threadIdx.x - POLICY_ROWS; it < POLICY_ROWS * NQ; it += POLICY_THREADS - POLICY_ROWS) {
            const int rr = it / NQ, q = it - rr * NQ;
            const int64_t r = base + rr;
            if (r >= n_rows) continue;
            const int64_t p = a.row_path ? (int64_t)a.row_path[r] : r;
            if (a.alive && !a.alive[p]) continue;
            const int64_t gid = a.path_ids ? (int64_t)a.path_ids[r] : a.path_base + p;
            const int a0 = q * 4, na = (A - a0) < 4 ? (A - a0) : 4;
            float z[4] = {0.f, 0.f, 0.f, 0.f};
            if (a.eps) {
                for (int k = 0; k < na; ++k) z[k] = a.eps[p * A + a0 + k];
            } else {                                   // one Philox block and two Box-Muller pairs per four values
                uint32_t o[4];
                philox4x32_10((uint32_t)gid, (uint32_t)((uint64_t)gid >> 32), (uint32_t)a.step,
                              ((uint32_t)RNG_STREAM_ACT << 16) | (uint32_t)q, (uint32_t)a.seed, (uint32_t)(a.seed >> 32), o);
                box_muller(o[0], o[1], z[0], z[1]);
                if (na > 2) box_muller(o[2], o[3], z[2], z[3]);
            }
            for (int k = 0; k < na; ++k) {
                const int i = a0 + k;
                const float mu = a.mu_raw[r * A + i];
                float pi;
                s_term[rr * A + i] = actor_dim<FAST>(mu, a.log_std[i], z[k], pi);
                s_pi[rr * A + i] = pi;
                if (a.pi) a.pi[r * A + i] = pi;
                if (a.mu) a.mu[r * A + i] = mu;
            }
        }
    }
    __syncthreads();
    if (threadIdx.x < POLICY_ROWS && s_live[threadIdx.x] && a.logp) {
        NpSumStream acc(A);
        for (int i = 0; i < A; ++i) acc.add(i, s_term[threadIdx.x * A + i]);
        a.logp[base + threadIdx.x] = acc.result();
    }
    if (!a.xin) return;                             // uniform over the block
    const int W = a.O + A;
    const int64_t left = n_rows - base;
    const int64_t nrows = left < 0 ? 0 : (left < POLICY_ROWS ? left : POLICY_ROWS);
    for (int idx = threadIdx.x; idx < nrows * W; idx += POLICY_THREADS) {
        const int rr = idx / W, c = idx - rr * W;
        if (!s_live[rr]) continue;
        a.xin[base * W + idx] = c < a.O ? a.obs[(base + rr) * a.O + c] : s_pi[rr * A + (c - a.O)];
    }
}

struct RawDyn {             // raw outputs [E, N, W]: row pointer of member 0 + member stride
    const float* row0; int64_t estride;
    __device__ RawDyn(const float* raw, int64_t N, int W, int64_t p) : row0(raw + p * W), estride(N * (int64_t)W) {}
    __device__ float operator()(int e, int c) const { return __ldg(row0 + (int64_t)e * estride + c); }
    __device__ const float* ptr(int c) const { return row0 + c; }      // member 0; member e at + e * estride
    __device__ static float load(const float* q) { return __ldg(q); }
};

struct RawStaged {          // the same rows staged in shared memory: [E, rows, W]
    const float* row0; int estride;
    __device__ RawStaged(const float* s_raw, int rows, int W, int r) : row0(s_raw + r * W), estride(rows * W) {}
    __device__ float operator()(int e, int c) const { return row0[e * estride + c]; }
    __device__ const float* ptr(int c) const { return row0 + c; }
    __device__ static float load(const float* q) { return *q; }
};

// ------------------------------------------------------------------------------------------------
// Dense row kernels: one thread per (row, obs dimension).  A block of 256 threads covers
// RB = 256 / O consecutive rows, so every lane is busy for any O (17, 29, 47 ...).  Phase 1 is the
// per-dimension arithmetic (env_dim, row_math.cuh); phase 2 runs on the row-owner thread (dim 0):
// ordered sums over the dimensions, statics, sampler rules, scalar writes; phase 3 writes the
// vector fields with all threads.
// ------------------------------------------------------------------------------------------------
constexpr int ROW_THREADS = 256;

struct RowShared {
    float kl[ROW_THREADS], epv[ROW_THREADS], nx[ROW_THREADS];
    unsigned char fin[ROW_THREADS], cut[ROW_THREADS];
    double stats[4];
};

struct EnvStepArgs {
    int64_t N; int O, A;
    EnvRowCfg c; int n_elite;
    const float* obs; const float* raw;   // raw [E,N,2D]
    const int32_t* elite_pos; const float* state_eps; const int32_t* path_ids;
    uint64_t seed; int step;
    float *next_obs, *rew, *cost; uint8_t* term; float *dkl_path, *ep_var;
    double* dkl_sum;   // 1 double accumulator
};

template <int EC, bool FAST>
__global__ void __launch_bounds__(ROW_THREADS, 4) env_step_kernel(EnvStepArgs a) {
    __shared__ RowShared sh;
    const int O = a.O, RB = ROW_THREADS / O;
    const int rb = threadIdx.x / O, dim = threadIdx.x - rb * O;
    if (threadIdx.x == 0) sh.stats[0] = 0.0;
    __syncthreads();
    for (int64_t base = (int64_t)blockIdx.x * RB; base < a.N; base += (int64_t)gridDim.x * RB) {
        const int64_t p = base + rb;
        const bool active = rb < RB && p < a.N;
        int member = 0;
        if (active) {
            const int64_t gid = a.path_ids ? (int64_t)a.path_ids[p] : p;
            const int pos = a.elite_pos ? a.elite_pos[p] : philox_elite_pos(a.seed, gid, a.step, a.n_elite);
            member = a.c.elite[pos];
            const float eps = (!a.c.deterministic && a.state_eps) ? a.state_eps[p * O + dim] : 1.0f;
            RawDyn raw(a.raw, a.N, 2 * a.c.D, p);
            EnvDimOut d = env_dim<EC, FAST>(a.c, raw, dim, member, a.obs[p * O + dim], eps);
            sh.kl[threadIdx.x] = d.kl; sh.epv[threadIdx.x] = d.epv; sh.nx[threadIdx.x] = d.nx;
            sh.fin[threadIdx.x] = isfinite(d.nx) ? 1 : 0;
            a.next_obs[p * O + dim] = d.nx;
            if (a.ep_var) a.ep_var[p * O + dim] = d.epv;
        }
        __syncthreads();
        if (active && dim == 0) {
            RawDyn raw(a.raw, a.N, 2 * a.c.D, p);
            EnvRowOut r = env_row_finish<FAST>(a.c, raw, member, sh.kl + rb * O, sh.epv + rb * O, sh.nx + rb * O,
                                         sh.fin + rb * O);
            a.rew[p] = r.rew; a.cost[p] = r.cost; a.term[p] = r.term ? 1 : 0;
            a.dkl_path[p] = r.dkl_path;
            atomicAdd(&sh.stats[0], (double)r.dkl_path);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0 && sh.stats[0] != 0.0) atomicAdd(a.dkl_sum, sh.stats[0]);   // fake_env.py:114
}

__global__ void finish_mean_kernel(const double* sum, int64_t n, float* out) {
    if (threadIdx.x == 0 && blockIdx.x == 0) out[0] = (float)(sum[0] / (double)n);
}

// ---- what a step does with one fed row once FakeEnv.step's outputs are known ---------------------
// sampler rules model_sampler.py:275-367 + ModelBuffer.store_multiple (modelbuffer.py:114-135)
struct StepRules {
    int64_t B; int t, last_storable;          // last_storable = T-2: storing it ends the path (horizon)
    int uncertainty; double dkl_lim;
    int no_store;                             // CMBPO_ROLLOUT_NO_STORE: per-path results and statistics only
    uint8_t* alive;                           // [B] by path
    uint8_t* pending;                         // [B] by path: bit0 last_val, bit1 last_cval wanted from the next policy pass
    cmbpo_rollout_bufs b;
};

struct RowCarry { float v, vc, logp; double dkl, ret, cost; };

// returns 1 = the step was stored, 2 = the path was cut as too uncertain BEFORE the store.
// st[0..3] += rows fed, sum dkl, rows stored, sum ep_var  (the caller reduces them per step)
__device__ __forceinline__ int step_row_commit(const StepRules& a, int64_t p, const EnvRowOut& o, const RowCarry& pf,
                                               double& st0, double& st1, double& st2, double& st3) {
    const float v = pf.v, vc = pf.vc;
    // uncertainty cut-off BEFORE the step is stored (model_sampler.py:275-290)
    const double next_dkl = pf.dkl + (double)o.dkl_path;
    const bool cut = a.uncertainty && next_dkl >= a.dkl_lim;
    st0 += 1.0; st1 += (double)o.dkl_path;
    if (cut) {
        a.alive[p] = 0;
        a.b.end_reason[p] = CMBPO_END_UNCERTAIN;
        a.b.last_val[p] = v; a.b.last_cval[p] = vc;      // V(s_t), VC(s_t): model_sampler.py:401-407
        return 2;
    }
    const int t = a.t;
    if (!a.no_store) {
        const int64_t row = (int64_t)t * a.B + p;      // ModelBuffer.store_multiple, time-major
        a.b.rew[row] = o.rew; a.b.val[row] = v; a.b.cost[row] = o.cost; a.b.cval[row] = vc;
        a.b.logp[row] = pf.logp; a.b.dyn_error[row] = o.ep_var_mean; a.b.dkl[row] = o.dkl_path;
        a.b.term[row] = o.term ? 1 : 0;
    }
    a.b.length[p] = t + 1;
    a.b.cum_dkl[p] = next_dkl;                        // model_sampler.py:332
    a.b.path_return[p] = pf.ret + (double)o.rew;      // :317-318
    a.b.path_cost[p] = pf.cost + (double)o.cost;
    st2 += 1.0; st3 += (double)o.ep_var_sum;
    if (t >= a.last_storable) {                       // path_length >= max_path_length-1 (:352)
        a.alive[p] = 0; a.b.end_reason[p] = CMBPO_END_HORIZON; a.pending[p] = 3;
    } else if (o.term) {                              // env terminal (:357-364)
        a.alive[p] = 0; a.b.end_reason[p] = CMBPO_END_TERMINAL;
        a.b.last_val[p] = 0.f; a.pending[p] = 2;
    }
    return 1;
}

// ---- rollout step ------------------------------------------------------------------------
struct StepArgs {
    StepRules rules;         // B, t, horizon / uncertainty rules, alive / pending flags, the buffers
    int64_t B; int O, A, T, t;
    EnvRowCfg c; int n_elite;
    int64_t path_base; uint64_t seed;
    const float* raw;        // [E,B,2D]
    float* cur_obs;          // [B,O] in/out
    uint8_t* alive;          // [B]
    const float *pi, *mu, *logp, *v, *vc;      // this step's policy outputs [B,..]
    const int32_t* elite_pos;                  // [B] slice for this step or null (indexed by path)
    const float* state_eps;                    // [B,O] slice or null (indexed by path)
    const int32_t* row_path;                   // [B] compact row -> path, or null (row == path)
    const int64_t* n_dev;                      // live row count (device), or null (B rows)
    cmbpo_rollout_bufs b;
};

// One block iteration handles `rows` = floor(512 / O) consecutive paths in phases that all run dense:
//   0: warp e stages member e's raw outputs [rows, 2D] (contiguous in global memory) into shared
//      memory with batches of 8 independent 8-byte loads per lane, so the DRAM / L2 latency is paid
//      twice per block instead of once per member and dimension; one thread per path draws the
//      elite member (Philox or injected)
//   1: one thread per (path, obs dim) -- member statistics, KL, next state (row_math.cuh)
//   2: one thread per path  -- ordered reductions over the dims, statics, sampler rules, the
//                              per-step scalars of ModelBuffer (coalesced: time-major rows)
//   3: one thread per (path, dim) -- obs / next_obs / act / mu rows, carried state
// (With phase 2 executed by the dim-0 thread of each path, as FakeEnv.step still does, a warp
// holds two paths and the serial part runs at 2/32 lane utilisation.)
constexpr int STEP_THREADS = 256;     // (128-thread blocks, 8 per SM, measured the same)
__host__ __device__ inline int step_rows(int O) { return 2 * STEP_THREADS / O < 64 ? 2 * STEP_THREADS / O : 64; }
__host__ __device__ inline size_t step_smem_bytes(int O, int E, int W) {
    const size_t rows = step_rows(O);
    return (size_t)E * rows * W * 4 + rows * O * (3 * sizeof(float) + 1) + rows * (2 * sizeof(int) + 1) + 16;
}

template <int EC, bool FAST>
__global__ void __launch_bounds__(STEP_THREADS, 4) rollout_step_kernel(StepArgs a) {
    extern __shared__ __align__(16) unsigned char step_smem[];
    const int O = a.O, A = a.A, t = a.t, E = a.c.E, W = 2 * a.c.D;
    const int rows = step_rows(O), NI = rows * O;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* s_raw = reinterpret_cast<float*>(step_smem);
    float* s_kl = s_raw + E * rows * W;
    float* s_epv = s_kl + NI;
    float* s_nx = s_epv + NI;
    int* s_member = reinterpret_cast<int*>(s_nx + NI);
    int* s_path = s_member + rows;
    unsigned char* s_fin = reinterpret_cast<unsigned char*>(s_path + rows);
    unsigned char* s_state = s_fin + NI;             // 0 = not fed, 1 = stored, 2 = cut
    __shared__ double s_stats[4];
    double st0 = 0.0, st1 = 0.0, st2 = 0.0, st3 = 0.0;   // rows fed, sum dkl, rows stored, sum ep_var
    if (threadIdx.x < 4) s_stats[threadIdx.x] = 0.0;
    // rows r of the (possibly compacted) batch: raw outputs, carried state and this step's policy outputs
    // are indexed by row; the ModelBuffer fields, alive / pending flags and injected noise by path
    const int64_t n_live = a.n_dev ? *a.n_dev : a.B;
    for (int64_t base = (int64_t)blockIdx.x * rows; base < n_live; base += (int64_t)gridDim.x * rows) {
        const int nrows = (n_live - base) < rows ? (int)(n_live - base) : rows;
        const int n2 = nrows * W / 2;                // W is even: 8-byte units, always aligned
        for (int e = warp; e < E; e += STEP_THREADS / 32) {
            const float2* src = reinterpret_cast<const float2*>(a.raw + ((int64_t)e * a.B + base) * W);
            float2* dst = reinterpret_cast<float2*>(s_raw + e * rows * W);
            for (int i0 = lane; i0 < n2; i0 += 32 * 8) {
                float2 v[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) if (i0 + 32 * k < n2) v[k] = __ldg(src + i0 + 32 * k);
#pragma unroll
                for (int k = 0; k < 8; ++k) if (i0 + 32 * k < n2) dst[i0 + 32 * k] = v[k];
            }
        }
        // the per-path scalars of phase 2 are fetched here, so their latency overlaps phases 0-1
        float pf_v = 0.f, pf_vc = 0.f, pf_logp = 0.f;
        double pf_dkl = 0.0, pf_ret = 0.0, pf_cost = 0.0;
        if (threadIdx.x < rows) {
            const int64_t r = base + threadIdx.x;
            int member = -1, path = -1;
            if (r < n_live) {
                path = a.row_path ? a.row_path[r] : (int)r;
                if (a.alive[path]) {
                    const int pos = a.elite_pos ? a.elite_pos[path] : philox_elite_pos(a.seed, a.path_base + path, t, a.n_elite);
                    member = a.c.elite[pos];
                    pf_v = a.v[r]; pf_vc = a.vc[r]; pf_logp = a.logp[r];
                    pf_dkl = a.b.cum_dkl[path]; pf_ret = a.b.path_return[path]; pf_cost = a.b.path_cost[path];
                }
            }
            s_member[threadIdx.x] = member;
            s_path[threadIdx.x] = path;
            s_state[threadIdx.x] = 0;
        }
        __syncthreads();
        for (int idx = threadIdx.x; idx < NI; idx += STEP_THREADS) {
            const int r = idx / O, dim = idx - r * O;
            const int member = s_member[r];
            if (member < 0) continue;
            const int64_t p = s_path[r];
            float eps = 1.0f;
            if (!a.c.deterministic)
                eps = a.state_eps ? a.state_eps[p * O + dim]
                                  : philox_normal(a.seed, a.path_base + p, t, RNG_STREAM_STATE, dim);
            RawStaged raw(s_raw, rows, W, r);
            const EnvDimOut d = env_dim<EC, FAST>(a.c, raw, dim, member, a.cur_obs[(base + r) * O + dim], eps);
            s_kl[idx] = d.kl; s_epv[idx] = d.epv; s_nx[idx] = d.nx;
            s_fin[idx] = isfinite(d.nx) ? 1 : 0;
        }
        __syncthreads();
        if (threadIdx.x < rows && s_member[threadIdx.x] >= 0) {
            const int r = threadIdx.x;
            const int64_t p = s_path[r];
            RawStaged raw(s_raw, rows, W, r);
            const EnvRowOut o = env_row_finish<FAST>(a.c, raw, s_member[r], s_kl + r * O, s_epv + r * O, s_nx + r * O,
                                               s_fin + r * O);
            RowCarry pf;
            pf.v = pf_v; pf.vc = pf_vc; pf.logp = pf_logp; pf.dkl = pf_dkl; pf.ret = pf_ret; pf.cost = pf_cost;
            s_state[r] = (unsigned char)step_row_commit(a.rules, p, o, pf, st0, st1, st2, st3);
        }
        __syncthreads();
        for (int idx = threadIdx.x; idx < NI; idx += STEP_THREADS) {
            const int r = idx / O, dim = idx - r * O;
            if (s_state[r] != 1) continue;
            const int64_t p = s_path[r], row = (int64_t)t * a.B + p;
            const float nx = s_nx[idx];
            if (!a.rules.no_store) {
                a.b.obs[row * O + dim] = a.cur_obs[(base + r) * O + dim];
                a.b.nextobs[row * O + dim] = nx;
            }
            a.cur_obs[(base + r) * O + dim] = nx;                 // model_sampler.py:350
        }
        if (!a.rules.no_store)
        for (int idx = threadIdx.x; idx < rows * A; idx += STEP_THREADS) {
            const int r = idx / A, i = idx - r * A;
            if (s_state[r] != 1) continue;
            const int64_t p = s_path[r], row = (int64_t)t * a.B + p;
            a.b.act[row * A + i] = a.pi[(base + r) * A + i];
            a.b.mu[row * A + i] = a.mu[(base + r) * A + i];
        }
        __syncthreads();
    }
    // per-step statistics: warp-reduce the row threads' partial sums, one shared atomic per warp
    if (threadIdx.x < 64) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            st0 += __shfl_down_sync(0xffffffffu, st0, off); st1 += __shfl_down_sync(0xffffffffu, st1, off);
            st2 += __shfl_down_sync(0xffffffffu, st2, off); st3 += __shfl_down_sync(0xffffffffu, st3, off);
        }
        if (lane == 0) {
            atomicAdd(&s_stats[0], st0); atomicAdd(&s_stats[1], st1);
            atomicAdd(&s_stats[2], st2); atomicAdd(&s_stats[3], st3);
        }
    }
    __syncthreads();
    if (threadIdx.x < 4 && s_stats[threadIdx.x] != 0.0)
        atomicAdd(a.b.step_stats + (int64_t)a.t * 4 + threadIdx.x, s_stats[threadIdx.x]);
}

__global__ void rollout_init_kernel(int64_t B, int O, const float* start, float* cur, uint8_t* alive,
                                    uint8_t* pending, cmbpo_rollout_bufs b) {
    int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= B) return;
    for (int o = 0; o < O; ++o) cur[p * O + o] = start[p * O + o];
    alive[p] = 1; pending[p] = 0;
    b.length[p] = 0; b.end_reason[p] = CMBPO_END_ALIVE;
    b.last_val[p] = 0.f; b.last_cval[p] = 0.f;
    b.cum_dkl[p] = 0.0; b.path_return[p] = 0.0; b.path_cost[p] = 0.0;
}

// paths still alive when the step budget ran out keep END_ALIVE; their bootstrap values are
// V(s_now), VC(s_now) so that finish_all_paths (model_sampler.py:418-444) is a no-op on the device
__global__ void rollout_final_kernel(int64_t B, int O, const float* cur, const uint8_t* alive,
                                     cmbpo_rollout_bufs b, const float* v, const float* vc,
                                     const int32_t* row_path, const int64_t* n_dev) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= (n_dev ? *n_dev : B)) return;
    const int64_t p = row_path ? (int64_t)row_path[r] : r;
    if (alive[p]) { b.last_val[p] = v[r]; b.last_cval[p] = vc[r]; }
    if (b.final_obs) for (int o = 0; o < O; ++o) b.final_obs[p * O + o] = cur[r * O + o];
}

// ---- alive-row compaction (tensor-core precisions, tasks / modes in which paths end early) ----------
// The reference only feeds the alive paths to the networks (model_sampler.py:255-259, 300-311).  Here
// the rows of finished paths are squeezed out of the batch every other step: flags -> exclusive scan
// (cmbpo_path_offsets) -> gather of the carried state and of the row -> path map; the row count
// lives in device memory and every kernel of the step reads it, so no host round trip is needed.
// A path that still waits for a bootstrap value (pending) stays one more policy pass.
__global__ void compact_init_kernel(int64_t B, int32_t* row_path, int64_t* n_dev) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < B) row_path[r] = (int32_t)r;
    if (r == 0) { n_dev[0] = B; n_dev[1] = B; }
}

__global__ void compact_flags_kernel(int64_t B, const int32_t* row_path, const int64_t* n_dev, const uint8_t* alive,
                                     const uint8_t* pending, int32_t* flags) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= B) return;
    int f = 0;
    if (r < *n_dev) { const int p = row_path[r]; f = (alive[p] || pending[p]) ? 1 : 0; }
    flags[r] = f;
}

__global__ void compact_gather_kernel(int64_t B, int O, const int32_t* flags, const int64_t* off, const int64_t* n_old,
                                      const float* cur, const int32_t* row_path, float* cur2, int32_t* row_path2,
                                      int64_t* n_new) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *n_new = off[B];
    const int64_t r = i / O;
    if (r >= *n_old || !flags[r]) return;
    const int c = (int)(i - r * O);
    const int64_t dst = off[r];
    cur2[dst * O + c] = cur[i];
    if (c == 0) row_path2[dst] = row_path[r];
}

EnvRowCfg make_env_cfg(const Net& dyn, const cmbpo_env_cfg& e, int O, int precision) {
    EnvRowCfg c;
    c.O = O; c.D = dyn.D; c.E = dyn.E;
    c.term_id = e.term_id; c.cost_id = e.cost_id; c.predicts_cost = e.predicts_cost;
    c.deterministic = e.deterministic; c.predicts_delta = e.predicts_delta;
    c.kl_closed_form = (precision != CMBPO_PREC_FP32) ? 1 : 0;
    c.sig_out = dyn.sig_out; c.mu_out = dyn.mu_out; c.l2s_out = dyn.l2s_out; c.elite = dyn.elite;
    return c;
}

ValueHead make_head(const Net& n, const float* raw) {
    ValueHead h;
    h.raw = raw; h.E = n.E; h.ld = 1;
    h.mu_out = n.has_out ? n.mu_out : nullptr; h.sig_out = n.sig_out;
    return h;
}

int check_dyn(const cmbpo_ctx* ctx, const cmbpo_env_cfg* cfg, int O) {
    const Net& dyn = ctx->nets[CMBPO_NET_DYN];
    CMBPO_CHECK(dyn.loaded && dyn.probabilistic, "dynamics ensemble not loaded (or not probabilistic)");
    CMBPO_CHECK(dyn.has_out, "dynamics ensemble needs an output scaler");
    CMBPO_CHECK(dyn.E <= CMBPO_MAX_E, "at most %d ensemble members", CMBPO_MAX_E);
    CMBPO_CHECK(O <= CMBPO_MAX_OBS, "obs dim %d > %d", O, CMBPO_MAX_OBS);
    CMBPO_CHECK(dyn.D == O + 1 + (cfg->predicts_cost ? 1 : 0), "model output width %d does not match obs dim %d", dyn.D, O);
    CMBPO_CHECK(dyn.n_elite > 0, "no elite indices");
    return 0;
}

// policy forward for N rows: actor MLP + V + VC chains, then the row kernel
int policy_forward(cmbpo_ctx* ctx, PolicyRowsArgs a, bool with_actor, int precision) {
    Net& actor = ctx->nets[CMBPO_NET_ACTOR];
    Net& v = ctx->nets[CMBPO_NET_V];
    Net& vc = ctx->nets[CMBPO_NET_VC];
    CMBPO_CHECK(v.loaded && vc.loaded, "value ensembles not loaded");
    if (precision != CMBPO_PREC_FP32 && ctx->polnet.loaded) {
        // tcgen05 path: actor + V + VC as ONE merged ensemble launch (policy_pack.cu)
        Net& pn = ctx->polnet;
        const int A = pn.dims[3];
        CMBPO_CHECK(ctx->log_std && A <= CMBPO_MAX_ACT, "actor not loaded");
        float* raw;
        if (cmbpo_ws_get(ctx, 3, (size_t)pn.E * a.N * A * sizeof(float), (void**)&raw)) return 1;
        if (ens_forward(ctx, pn, a.obs, a.N, false, raw, precision, a.n_dev)) return 1;
        a.mu_raw = with_actor ? raw : nullptr;
        a.log_std = ctx->log_std;
        a.v = make_head(v, raw + (size_t)a.N * A); a.v.ld = A;
        a.vc = make_head(vc, raw + (size_t)(1 + v.E) * a.N * A); a.vc.ld = A;
        policy_rows_kernel<true><<<cdiv(a.N, POLICY_ROWS), POLICY_THREADS, 0, ctx->stream>>>(a);
        ctx->launches++;
        CUDA_TRY(cudaGetLastError());
        return 0;
    }
    float *raw_v, *raw_vc, *raw_mu = nullptr;
    if (cmbpo_ws_get(ctx, 3, (size_t)(v.E + vc.E) * a.N * sizeof(float), (void**)&raw_v)) return 1;
    raw_vc = raw_v + (size_t)v.E * a.N;
    // small nets: tcgen05 path only if supported, else fp32 (decided per net: V and VC may differ in shape)
    const int pv = (precision != CMBPO_PREC_FP32 && ens_tc_supported(v)) ? precision : CMBPO_PREC_FP32;
    const int pvc = (precision != CMBPO_PREC_FP32 && ens_tc_supported(vc)) ? precision : CMBPO_PREC_FP32;
    if (ens_forward(ctx, v, a.obs, a.N, false, raw_v, pv)) return 1;
    if (ens_forward(ctx, vc, a.obs, a.N, false, raw_vc, pvc)) return 1;
    if (with_actor) {
        CMBPO_CHECK(actor.loaded && ctx->log_std, "actor not loaded");
        CMBPO_CHECK(a.A <= CMBPO_MAX_ACT, "act dim too large");
        if (cmbpo_ws_get(ctx, 4, (size_t)a.N * a.A * sizeof(float), (void**)&raw_mu)) return 1;
        int pa = (precision != CMBPO_PREC_FP32 && ens_tc_supported(actor)) ? precision : CMBPO_PREC_FP32;
        if (ens_forward(ctx, actor, a.obs, a.N, false, raw_mu, pa)) return 1;
    }
    a.mu_raw = raw_mu; a.log_std = ctx->log_std;
    a.v = make_head(v, raw_v); a.vc = make_head(vc, raw_vc);
    if (precision != CMBPO_PREC_FP32) policy_rows_kernel<true><<<cdiv(a.N, POLICY_ROWS), POLICY_THREADS, 0, ctx->stream>>>(a);
    else policy_rows_kernel<false><<<cdiv(a.N, POLICY_ROWS), POLICY_THREADS, 0, ctx->stream>>>(a);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

}  // namespace

extern "C" int cmbpo_policy_act(cmbpo_ctx* ctx, const float* obs, int64_t N, const float* eps,
                                const int32_t* path_ids, uint64_t seed, int step, float* pi,
                                float* logp, float* mu, float* v, float* vc, int precision) {
    CMBPO_CHECK(ctx, "null context");
    if (N <= 0) return 0;
    Net& actor = ctx->nets[CMBPO_NET_ACTOR];
    const bool with_actor = (pi != nullptr || mu != nullptr || logp != nullptr);
    PolicyRowsArgs a = {};
    a.N = N; a.O = ctx->nets[CMBPO_NET_V].dims[0]; a.A = with_actor ? actor.dims[actor.n_layers] : 0;
    a.obs = obs; a.eps = eps; a.path_ids = path_ids; a.path_base = 0; a.seed = seed; a.step = step;
    a.pi = pi; a.logp = logp; a.mu = mu; a.vout = v; a.vcout = vc;
    return policy_forward(ctx, a, with_actor, precision);
}

extern "C" int cmbpo_fakeenv_step(cmbpo_ctx* ctx, const cmbpo_env_cfg* cfg, const float* obs,
                                  const float* act, int64_t N, const int32_t* elite_pos,
                                  const float* state_eps, const int32_t* path_ids, uint64_t seed,
                                  int step, float* next_obs, float* rew, float* cost, uint8_t* term,
                                  float* dkl_path, float* ep_var, float* dkl_mean_out, int precision) {
    CMBPO_CHECK(ctx && cfg, "null argument");
    if (N <= 0) return 0;
    Net& dyn = ctx->nets[CMBPO_NET_DYN];
    CMBPO_CHECK(dyn.loaded, "dynamics ensemble not loaded");
    const int Din = dyn.dims[0];
    const int O = dyn.D - 1 - (cfg->predicts_cost ? 1 : 0), A = Din - O;
    if (check_dyn(ctx, cfg, O)) return 1;
    // concat(obs, act) (fake_env.py:81)
    float *xin, *raw;
    double* dsum;
    if (cmbpo_ws_get(ctx, 4, (size_t)N * Din * sizeof(float) + 64, (void**)&xin)) return 1;
    dsum = (double*)((char*)xin + (((size_t)N * Din * sizeof(float) + 15) / 16) * 16);
    CUDA_TRY(cudaMemcpy2DAsync(xin, Din * sizeof(float), obs, O * sizeof(float), O * sizeof(float), N,
                               cudaMemcpyDeviceToDevice, ctx->stream));
    CUDA_TRY(cudaMemcpy2DAsync(xin + O, Din * sizeof(float), act, A * sizeof(float), A * sizeof(float),
                               N, cudaMemcpyDeviceToDevice, ctx->stream));
    CUDA_TRY(cudaMemsetAsync(dsum, 0, sizeof(double), ctx->stream));
    if (cmbpo_ws_get(ctx, 2, (size_t)dyn.E * N * 2 * dyn.D * sizeof(float), (void**)&raw)) return 1;
    if (ens_forward(ctx, dyn, xin, N, false, raw, precision)) return 1;
    EnvStepArgs a = {};
    a.N = N; a.O = O; a.A = A; a.c = make_env_cfg(dyn, *cfg, O, precision); a.n_elite = dyn.n_elite;
    a.obs = obs; a.raw = raw; a.elite_pos = elite_pos; a.state_eps = state_eps; a.path_ids = path_ids;
    a.seed = seed; a.step = step;
    a.next_obs = next_obs; a.rew = rew; a.cost = cost; a.term = term; a.dkl_path = dkl_path;
    a.ep_var = ep_var; a.dkl_sum = dsum;
    {
        const int grid = min(cdiv(N, ROW_THREADS / O), ctx->sm_count * 16);
        if (a.c.kl_closed_form && a.c.E == 7) env_step_kernel<7, true><<<grid, ROW_THREADS, 0, ctx->stream>>>(a);
        else { a.c.kl_closed_form = 0; env_step_kernel<0, false><<<grid, ROW_THREADS, 0, ctx->stream>>>(a); }
    }
    if (dkl_mean_out) finish_mean_kernel<<<1, 32, 0, ctx->stream>>>(dsum, N, dkl_mean_out);
    ctx->launches += 2;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int cmbpo_rollout(cmbpo_ctx* ctx, const cmbpo_rollout_cfg* cfg, const cmbpo_rollout_bufs* bufs) {
    CMBPO_CHECK(ctx && cfg && bufs, "null argument");
    const int64_t B = cfg->B;
    if (B <= 0) return 0;
    Net& dyn = ctx->nets[CMBPO_NET_DYN];
    Net& actor = ctx->nets[CMBPO_NET_ACTOR];
    CMBPO_CHECK(dyn.loaded && actor.loaded, "networks not loaded");
    const int Din = dyn.dims[0];
    const int A = actor.dims[actor.n_layers], O = Din - A;
    if (check_dyn(ctx, &cfg->env, O)) return 1;
    const int T = cfg->T;
    CMBPO_CHECK(T >= 2, "max_path_length must be >= 2");
    const int n_steps = (cfg->max_steps > 0 && cfg->max_steps < T - 1) ? cfg->max_steps : T - 1;

    float *cur, *cur2, *pi, *mu, *logp, *v, *vc, *xin, *raw;
    uint8_t *alive, *pending;
    int32_t *row_path[2], *cflags;
    int64_t *n_dev, *coff;
    size_t fl = (size_t)B * (2 * O + 2 * A + 3 + Din);
    char* base;
    // floats | int64 (2 row counts + B+1 scan offsets) | int32 (2 row maps + flags) | bytes
    const size_t bytes_f = fl * sizeof(float), bytes_l = ((size_t)B + 4) * sizeof(int64_t), bytes_i = 3 * (size_t)B * sizeof(int32_t);
    if (cmbpo_ws_get(ctx, 5, bytes_f + bytes_l + bytes_i + 2 * (size_t)B + 256, (void**)&base)) return 1;
    cur = (float*)base; cur2 = cur + (size_t)B * O; pi = cur2 + (size_t)B * O; mu = pi + (size_t)B * A; logp = mu + (size_t)B * A;
    v = logp + B; vc = v + B; xin = vc + B;
    char* q = base + ((bytes_f + 15) & ~(size_t)15);
    n_dev = (int64_t*)q; coff = n_dev + 2;
    row_path[0] = (int32_t*)(q + bytes_l); row_path[1] = row_path[0] + B; cflags = row_path[1] + B;
    alive = (uint8_t*)(cflags + B); pending = alive + B;
    // alive-row compaction: only where paths can end before the horizon, and only on the tcgen05 path
    // (the fp32 GEMM kernels take their row count from the host)
    const bool compacting = cfg->precision != CMBPO_PREC_FP32 && !(cfg->flags & CMBPO_ROLLOUT_NO_COMPACT) &&
                            (cfg->uncertainty_mode || cfg->env.term_id != CMBPO_TERM_NO_DONE);
    int cur_gen = 0;
    const int compact_every = cfg->compact_every > 0 ? cfg->compact_every : 2;    // measured: 2 beats 1 and 4 by 2-6 %
    if (cmbpo_ws_get(ctx, 2, (size_t)dyn.E * B * 2 * dyn.D * sizeof(float), (void**)&raw)) return 1;

    CUDA_TRY(cudaMemsetAsync(bufs->step_stats, 0, (size_t)T * 4 * sizeof(double), ctx->stream));
    rollout_init_kernel<<<cdiv(B, 256), 256, 0, ctx->stream>>>(B, O, bufs->start_obs, cur, alive, pending, *bufs);
    ctx->launches++;
    if (compacting) {
        compact_init_kernel<<<cdiv(B, 256), 256, 0, ctx->stream>>>(B, row_path[0], n_dev);
        ctx->launches++;
        if (!ctx->host_n) {
            CUDA_TRY(cudaHostAlloc((void**)&ctx->host_n, 4 * sizeof(int64_t), cudaHostAllocDefault));
            for (cudaEvent_t& e : ctx->n_ev) CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        }
    }
    // The live row count is mirrored to the host after every compaction; the host stays at most 3
    // compactions (6 steps = 24 launches) ahead of the device and stops issuing steps once no path is
    // alive or waiting for a bootstrap value (short rollouts in 'uncertainty' mode end long before the
    // horizon, and 30 steps of empty launches cost more than the steps that did work).
    int n_compactions = 0;

    for (int t = 0; t <= n_steps; ++t) {
        const bool last = (t == n_steps);
        if (compacting && n_compactions >= 3) {
            const int slot = (n_compactions - 3) & 3;          // the compaction three back
            CUDA_TRY(cudaEventSynchronize(ctx->n_ev[slot]));
            if (ctx->host_n[slot] == 0) break;                 // nothing alive, nothing pending
        }
        PolicyRowsArgs pa = {};
        pa.N = B; pa.O = O; pa.A = A; pa.obs = cur;
        pa.row_path = compacting ? row_path[cur_gen] : nullptr;
        pa.n_dev = compacting ? n_dev + cur_gen : nullptr;
        pa.eps = (bufs->act_eps && !last) ? bufs->act_eps + (size_t)t * B * A : nullptr;
        pa.path_base = cfg->path_id_base; pa.seed = cfg->seed; pa.step = t;
        pa.alive = alive; pa.pi = pi; pa.logp = logp; pa.mu = mu; pa.vout = v; pa.vcout = vc;
        pa.xin = xin; pa.pending = pending; pa.last_val = bufs->last_val; pa.last_cval = bufs->last_cval;
        {
            ProfScope prof(ctx, CMBPO_PROF_POLICY);
            if (policy_forward(ctx, pa, !last, cfg->precision)) return 1;
        }
        if (last) break;
        if (ens_forward(ctx, dyn, xin, B, false, raw, cfg->precision, pa.n_dev)) return 1;
        StepArgs sa = {};
        sa.row_path = pa.row_path; sa.n_dev = pa.n_dev;
        sa.B = B; sa.O = O; sa.A = A; sa.T = T; sa.t = t;
        sa.c = make_env_cfg(dyn, cfg->env, O, cfg->precision); sa.n_elite = dyn.n_elite;
        sa.rules.B = B; sa.rules.t = t; sa.rules.last_storable = T - 2;
        sa.rules.uncertainty = cfg->uncertainty_mode; sa.rules.dkl_lim = cfg->dkl_lim;
        sa.rules.alive = alive; sa.rules.pending = pending; sa.rules.b = *bufs;
        sa.rules.no_store = (cfg->flags & CMBPO_ROLLOUT_NO_STORE) ? 1 : 0;
        sa.path_base = cfg->path_id_base; sa.seed = cfg->seed;
        sa.raw = raw; sa.cur_obs = cur; sa.alive = alive;
        sa.pi = pi; sa.mu = mu; sa.logp = logp; sa.v = v; sa.vc = vc;
        sa.elite_pos = bufs->elite_pos ? bufs->elite_pos + (size_t)t * B : nullptr;
        sa.state_eps = bufs->state_eps ? bufs->state_eps + (size_t)t * B * O : nullptr;
        sa.b = *bufs;
        {
            const size_t smem = step_smem_bytes(O, dyn.E, 2 * dyn.D);
            const bool fast = sa.c.kl_closed_form && sa.c.E == 7;
            if (!fast) sa.c.kl_closed_form = 0;      // other ensemble sizes: the exact (all-pairs) variant
            auto kern = fast ? rollout_step_kernel<7, true> : rollout_step_kernel<0, false>;
            if (smem > ctx->step_smem_max[fast]) {
                CMBPO_CHECK(smem <= 200 * 1024, "rollout step: obs dim / ensemble too large for the staging buffer");
                CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                ctx->step_smem_max[fast] = smem;
            }
            ProfScope prof(ctx, CMBPO_PROF_STEP);
            kern<<<(unsigned)std::min<int64_t>(cdiv(B, step_rows(O)), (int64_t)ctx->sm_count * 64), STEP_THREADS, smem, ctx->stream>>>(sa);
        }
        ctx->launches++;
        if (compacting && (t % compact_every) == compact_every - 1 && t + 1 < n_steps) {
            compact_flags_kernel<<<cdiv(B, 256), 256, 0, ctx->stream>>>(B, row_path[cur_gen], n_dev + cur_gen, alive, pending, cflags);
            ctx->launches++;
            if (cmbpo_path_offsets(ctx, cflags, B, coff)) return 1;
            compact_gather_kernel<<<cdiv(B * O, 256), 256, 0, ctx->stream>>>(B, O, cflags, coff, n_dev + cur_gen, cur,
                                                                            row_path[cur_gen], cur2, row_path[cur_gen ^ 1],
                                                                            n_dev + (cur_gen ^ 1));
            ctx->launches++;
            std::swap(cur, cur2);
            cur_gen ^= 1;
            const int slot = n_compactions & 3;
            CUDA_TRY(cudaMemcpyAsync(ctx->host_n + slot, n_dev + cur_gen, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
            CUDA_TRY(cudaEventRecord(ctx->n_ev[slot], ctx->stream));
            ++n_compactions;
        }
    }
    rollout_final_kernel<<<cdiv(B, 256), 256, 0, ctx->stream>>>(B, O, cur, alive, *bufs, v, vc,
                                                                 compacting ? row_path[cur_gen] : nullptr,
                                                                 compacting ? n_dev + cur_gen : nullptr);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// ---- batch-global truncation --------------------------------------------------------------
namespace {

__global__ void hist_kernel(const int32_t* length, const uint8_t* reason, int64_t B, int T,
                            unsigned long long* hist) {
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < B;
         p += (int64_t)gridDim.x * blockDim.x) {
        int L = length[p];
        if (L < 0) L = 0;
        if (L > T) L = T;
        atomicAdd(hist + L, 1ull);
        if (reason[p] == CMBPO_END_UNCERTAIN) atomicAdd(hist + (T + 1) + L, 1ull);
    }
}

__global__ void cap_flags_kernel(const int32_t* length, int64_t B, int cap_step, int32_t* flags) {
    int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < B) flags[p] = length[p] > cap_step ? 1 : 0;
}

// close path p at step s with V(s_s), VC(s_s) = val[s][p], cval[s][p]
__device__ __forceinline__ void cut_path(const cmbpo_rollout_bufs& b, int64_t B, int64_t p, int s,
                                         int reason) {
    b.length[p] = s;
    b.end_reason[p] = (uint8_t)reason;
    b.last_val[p] = b.val[(int64_t)s * B + p];
    b.last_cval[p] = b.cval[(int64_t)s * B + p];
}

__global__ void cap_apply_kernel(cmbpo_rollout_bufs b, int64_t B, int cap_step, int64_t cap_n,
                                 const int64_t* rank) {
    int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= B) return;
    if (b.length[p] > cap_step && rank[p] < cap_n) cut_path(b, B, p, cap_step, CMBPO_END_CAPPED);
}

__global__ void stop_apply_kernel(cmbpo_rollout_bufs b, int64_t B, int stop_step) {
    int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= B) return;
    if (b.length[p] > stop_step + 1) cut_path(b, B, p, stop_step + 1, CMBPO_END_STOPPED);
}


// Diagnostics of a finished rollout over the VALID steps (t < length[p]) in one pass: one thread per
// path walks its steps in time order (time-major buffers: coalesced across paths), float64 sums.
//   stats[0..4] = sum rew, cost, val, cval, dyn_error;  stats[5] = max dkl;
//   stats[6] = max over (p, t) of the running return sum_{s<=t} rew;  stats[7] = number of steps
__global__ void rollout_diag_kernel(cmbpo_rollout_bufs b, int64_t B, double* path_return, double* path_cost,
                                    double* stats) {
    double s[5] = {0, 0, 0, 0, 0}, mx_dkl = -1e300, mx_ret = -1e300, n = 0;
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < B; p += (int64_t)gridDim.x * blockDim.x) {
        const int len = b.length[p];
        double pr = 0, pc = 0;
        for (int t = 0; t < len; ++t) {
            const int64_t i = (int64_t)t * B + p;
            const double r = (double)b.rew[i], c = (double)b.cost[i];
            pr += r; pc += c;
            s[2] += (double)b.val[i]; s[3] += (double)b.cval[i]; s[4] += (double)b.dyn_error[i];
            mx_dkl = fmax(mx_dkl, (double)b.dkl[i]);
            mx_ret = fmax(mx_ret, pr);
        }
        s[0] += pr; s[1] += pc; n += len;
        path_return[p] = pr; path_cost[p] = pc;
    }
    __shared__ double sh[8][8];
    double v[8] = {s[0], s[1], s[2], s[3], s[4], mx_dkl, mx_ret, n};
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const bool is_max = (k == 5 || k == 6);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const double o = __shfl_down_sync(0xffffffffu, v[k], off);
            v[k] = is_max ? fmax(v[k], o) : v[k] + o;
        }
        if ((threadIdx.x & 31) == 0) sh[k][threadIdx.x >> 5] = v[k];
    }
    __syncthreads();
    if (threadIdx.x < 8) {
        const int k = threadIdx.x;
        const bool is_max = (k == 5 || k == 6);
        double a = sh[k][0];
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) a = is_max ? fmax(a, sh[k][w]) : a + sh[k][w];
        if (!is_max) atomicAdd(stats + k, a);
        else {      // float64 max through the ordered-integer image (both signs)
            long long ai = __double_as_longlong(a);
            ai = ai >= 0 ? ai : (ai ^ 0x7fffffffffffffffLL);
            atomicMax(reinterpret_cast<long long*>(stats) + k, ai);
        }
    }
}

__global__ void rollout_diag_finish_kernel(double* stats) {
    const int k = 5 + threadIdx.x;             // decode the two maxima
    if (threadIdx.x < 2) {
        long long ai = reinterpret_cast<long long*>(stats)[k];
        ai = ai >= 0 ? ai : (ai ^ 0x7fffffffffffffffLL);
        stats[k] = __longlong_as_double(ai);
    }
}
}  // namespace

extern "C" int cmbpo_rollout_histogram(cmbpo_ctx* ctx, const int32_t* length, const uint8_t* end_reason,
                                       int64_t B, int T, int64_t* hist_host) {
    CMBPO_CHECK(ctx && hist_host, "null argument");
    unsigned long long* d;
    size_t bytes = 2 * (size_t)(T + 1) * sizeof(unsigned long long);
    if (cmbpo_ws_get(ctx, 6, bytes, (void**)&d)) return 1;
    CUDA_TRY(cudaMemsetAsync(d, 0, bytes, ctx->stream));
    hist_kernel<<<max(1, min(ctx->sm_count * 4, cdiv(B, 256))), 256, 0, ctx->stream>>>(length, end_reason, B, T, d);
    ctx->launches++;
    CUDA_TRY(cudaMemcpyAsync(hist_host, d, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int cmbpo_rollout_diagnostics(cmbpo_ctx* ctx, const cmbpo_rollout_bufs* bufs, int64_t B,
                                         double* path_return, double* path_cost, double* stats_host) {
    CMBPO_CHECK(ctx && bufs && path_return && path_cost && stats_host, "null argument");
    double* d;
    if (cmbpo_ws_get(ctx, 6, 8 * sizeof(double), (void**)&d)) return 1;
    // sums start at 0; the maxima at the ordered-integer image of -inf
    double init[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long ninf; { const double x = -1e300; memcpy(&ninf, &x, 8); ninf = ninf >= 0 ? ninf : (ninf ^ 0x7fffffffffffffffLL); }
    memcpy(&init[5], &ninf, 8); memcpy(&init[6], &ninf, 8);
    CUDA_TRY(cudaMemcpyAsync(d, init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));          // `init` is a stack buffer
    if (B > 0) {
        rollout_diag_kernel<<<max(1, min(ctx->sm_count * 8, cdiv(B, 256))), 256, 0, ctx->stream>>>(*bufs, B, path_return, path_cost, d);
        ctx->launches++;
    }
    rollout_diag_finish_kernel<<<1, 32, 0, ctx->stream>>>(d);
    ctx->launches++;
    CUDA_TRY(cudaMemcpyAsync(stats_host, d, 8 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int cmbpo_rollout_truncate(cmbpo_ctx* ctx, const cmbpo_rollout_bufs* bufs, int64_t B, int T,
                                      int cap_step, int64_t cap_n, int stop_step) {
    CMBPO_CHECK(ctx && bufs, "null argument");
    (void)T;
    if (cap_step >= 0 && cap_n > 0) {
        int32_t* flags;
        int64_t* rank;
        char* base;
        if (cmbpo_ws_get(ctx, 4, (size_t)B * 4 + (size_t)(B + 1) * 8 + 64, (void**)&base)) return 1;
        rank = (int64_t*)base;
        flags = (int32_t*)(base + (size_t)(B + 1) * 8);
        cap_flags_kernel<<<cdiv(B, 256), 256, 0, ctx->stream>>>(bufs->length, B, cap_step, flags);
        ctx->launches++;
        if (cmbpo_path_offsets(ctx, flags, B, rank)) return 1;
        cap_apply_kernel<<<cdiv(B, 256), 256, 0, ctx->stream>>>(*bufs, B, cap_step, cap_n, rank);
        ctx->launches++;
    }
    if (stop_step >= 0) {
        stop_apply_kernel<<<cdiv(B, 256), 256, 0, ctx->stream>>>(*bufs, B, stop_step);
        ctx->launches++;
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}
