// Per-row arithmetic of the rollout step and of the single FakeEnv step (rollout.cu).  The fp32 and
// the tensor-core precision modes run the same code; the FAST template argument selects the
// tensor-core modes' approximate divisions and closed-form KL.
//
// Everything here follows the reference's op order in float32 without FMA contraction
// (__fmul_rn / __fadd_rn), because numpy/TF evaluate these expressions one ufunc at a time.
#pragma once
#include "common.cuh"

// ------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011).  Counter = (path id lo, path id hi, step, stream<<16|block),
// key = seed.  Keyed by GLOBAL path id so results do not depend on how paths are sharded.
// ------------------------------------------------------------------------------------------
enum { RNG_STREAM_ACT = 0, RNG_STREAM_ELITE = 1, RNG_STREAM_STATE = 2 };

__host__ __device__ inline void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                              uint32_t k0, uint32_t k1, uint32_t out[4]) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += W0; k1 += W1;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// two standard normals from two uint32 (Box-Muller on (u+0.5)/2^32)
__device__ inline void box_muller(uint32_t a, uint32_t b, float& z0, float& z1) {
    float u1 = ((float)a + 0.5f) * 2.3283064365386963e-10f;
    float u2 = ((float)b + 0.5f) * 2.3283064365386963e-10f;
    u1 = fminf(u1, 0.99999994f);
    float r = sqrtf(-2.0f * logf(u1));
    float s, c;
    sincospif(2.0f * u2, &s, &c);
    z0 = r * c;
    z1 = r * s;
}

// the k-th standard normal of (path, step, stream)
__device__ inline float philox_normal(uint64_t seed, int64_t path, int step, int stream, int k) {
    uint32_t o[4];
    philox4x32_10((uint32_t)path, (uint32_t)((uint64_t)path >> 32), (uint32_t)step,
                  ((uint32_t)stream << 16) | (uint32_t)(k >> 2), (uint32_t)seed,
                  (uint32_t)(seed >> 32), o);
    float z0, z1;
    if ((k & 3) < 2) box_muller(o[0], o[1], z0, z1); else box_muller(o[2], o[3], z0, z1);
    return (k & 1) ? z1 : z0;
}

// uniform elite position in [0, n_elite): what np.random.choice(elite_inds, N) draws (fake_env.py:176)
__device__ inline int philox_elite_pos(uint64_t seed, int64_t path, int step, int n_elite) {
    uint32_t o[4];
    philox4x32_10((uint32_t)path, (uint32_t)((uint64_t)path >> 32), (uint32_t)step,
                  ((uint32_t)RNG_STREAM_ELITE << 16), (uint32_t)seed, (uint32_t)(seed >> 32), o);
    return (int)(((uint64_t)o[0] * (uint64_t)n_elite) >> 32);
}

// ------------------------------------------------------------------------------------------
// numpy's float32 pairwise sum for n < 128 elements (np.mean over the last axis):
// 8 running partial sums, a fixed combination tree, then the n%8 tail added sequentially.
// ------------------------------------------------------------------------------------------
__device__ inline float np_sum(const float* a, int n) {
    if (n < 8) {
        float s = 0.f;
        for (int i = 0; i < n; ++i) s = __fadd_rn(s, a[i]);
        return s;
    }
    float r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = a[j];
    int i = 8;
    for (; i < n - (n & 7); i += 8) {
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = __fadd_rn(r[j], a[i + j]);
    }
    float s = __fadd_rn(__fadd_rn(__fadd_rn(r[0], r[1]), __fadd_rn(r[2], r[3])),
                        __fadd_rn(__fadd_rn(r[4], r[5]), __fadd_rn(r[6], r[7])));
    for (; i < n; ++i) s = __fadd_rn(s, a[i]);
    return s;
}

// Streaming form of the same order: elements arrive one by one (i = 0 .. n-1), the partial sums stay
// in registers (all indices static after unrolling), so a per-row loop needs no local-memory array.
struct NpSumStream {
    float r[8], s;
    int n, nb;                       // nb = n - n % 8: elements before the sequential tail
    __device__ explicit NpSumStream(int n_) : s(0.f), n(n_), nb(n_ - (n_ & 7)) {
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = 0.f;
    }
    __device__ __forceinline__ void tree() {
        s = __fadd_rn(__fadd_rn(__fadd_rn(r[0], r[1]), __fadd_rn(r[2], r[3])),
                      __fadd_rn(__fadd_rn(r[4], r[5]), __fadd_rn(r[6], r[7])));
    }
    __device__ __forceinline__ void add(int i, float x) {
        if (n < 8) { s = __fadd_rn(s, x); return; }
        if (i < nb) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if ((i & 7) == j) r[j] = (i < 8) ? x : __fadd_rn(r[j], x);
            if (i == nb - 1) tree();
        } else {
            s = __fadd_rn(s, x);
        }
    }
    __device__ __forceinline__ float result() const { return s; }
};

// ------------------------------------------------------------------------------------------
// FakeEnv.step for one row (fake_env.py:104-153) given the raw last-layer outputs of all E
// members.  `raw(e, c)` returns column c of member e for this row (c < 2*D).
// ------------------------------------------------------------------------------------------
struct EnvRowCfg {
    int O, D, E;                 // D = O + 1 (+1 if the model predicts the cost)
    int term_id, cost_id, predicts_cost, deterministic, predicts_delta;
    int kl_closed_form;          // 1: O(E) closed form of the pairwise KL sum (tensor-core precision modes)
    const float* sig_out;        // [D] max(sqrt(var),1e-2)   (pens/utils.py:167)
    const float* mu_out;         // [D]
    const float* l2s_out;        // [D] 2*log(sigma)          (pens/utils.py:187)
    const int* elite;            // [n_elite]
};

struct EnvRowOut {
    float rew, cost, dkl_path, ep_var_mean, ep_var_sum;
    bool term;
};

// ------------------------------------------------------------------------------------------
// Gaussian actor head for one row (ac_network.py:105-111, 46-48)
// ------------------------------------------------------------------------------------------
// One action dimension: pi = mu + eps * exp(log_std) (ac_network.py:109) and its log-likelihood term
// (ac_network.py:47).  FAST (tensor-core precision modes): approximate division (2 ulp) -- the IEEE
// division is a subroutine call per use.
template <bool FAST>
__device__ __forceinline__ float actor_dim(float mu, float ls, float eps, float& pi) {
    const float log2pi = 1.8378770664093453f;   // float32(np.log(2*np.pi))
    const float sd = expf(ls);
    pi = __fadd_rn(mu, __fmul_rn(eps, sd));
    const float num = __fsub_rn(pi, mu), den = __fadd_rn(sd, 1e-8f);
    const float z = FAST ? __fdividef(num, den) : __fdiv_rn(num, den);
    const float t = __fadd_rn(__fadd_rn(__fmul_rn(z, z), __fmul_rn(2.0f, ls)), log2pi);
    return __fmul_rn(-0.5f, t);
}

// ------------------------------------------------------------------------------------------
// FakeEnv.step split per (row, obs dimension) -- the unit of work of the dense row kernels.
// env_dim: everything that only needs the E members' outputs for ONE dimension
// (fake_env.py:104-113 for that column); env_row_finish: the reductions over dimensions, statics,
// reward (fake_env.py:113-153).
//
// Arithmetic notes.  mean / next_obs / ep_var follow the reference's float32 op order exactly.
// The KL term uses two algebraic shortcuts that change results only at rounding level (tests
// state rtol 2e-3 on dkl): log_std = logvar/2 and exp(2 log_std) = var instead of
// log(sqrt(exp(logvar))) round trips (with the reference's clip behaviour kept for var == 0 / inf),
// and multiplication by a per-member reciprocal instead of 49 IEEE divisions.
// ------------------------------------------------------------------------------------------
struct EnvDimOut { float kl, epv, nx; };

// EC > 0: ensemble size known at compile time (loops fully unrolled, no predicates); EC == 0: runtime E.
// FAST (the tensor-core precision modes): closed-form KL and approximate divisions (2 ulp) -- the IEEE
// division is a subroutine call per use, and the all-pairs loop is 49 x 12 instructions of code.
// Kernels are instantiated for (EC = 7, FAST) -- the 7-member ensemble of every config in the
// tensor-core precision modes -- and for (EC = 0, exact): runtime E, IEEE divisions, all-pairs KL.
template <int EC, bool FAST, class Raw>
__device__ __forceinline__ EnvDimOut env_dim(const EnvRowCfg& c, Raw raw, int o, int member, float obs_o, float eps) {
    constexpr int EMAX = EC > 0 ? EC : CMBPO_MAX_E;
    const int E = EC > 0 ? EC : c.E;
    float nd[EMAX], ls[EMAX], vr[EMAX], rv[EMAX];
    const float sg = c.sig_out[o], mu = c.mu_out[o], l2s = c.l2s_out[o];
    float sel = 0.f;
    // two running pointers (mean column, log-variance column) advanced by the member stride
    const float* pm = raw.ptr(o);
    const float* pv = raw.ptr(c.D + o);
    const auto es = raw.estride;
#pragma unroll
    for (int e = 0; e < EMAX; ++e) {
        if (e < E) {
            const float mean = __fadd_rn(__fmul_rn(sg, raw.load(pm)), mu);        // pe.py:815-821
            const float logvar = __fadd_rn(l2s, raw.load(pv));                    // pe.py:826-828
            pm += es; pv += es;
            const float var = FAST ? __expf(logvar) : expf(logvar);               // pe.py:833
            float x = mean;
            if (!c.deterministic) {                                              // fake_env.py:104-106
                // FAST: var * rsqrt(var) (2 ulp) -- the IEEE square root is a subroutine call
                const float sd = FAST ? ((var > 0.f && !isinf(var)) ? __fmul_rn(var, rsqrtf(var)) : var) : sqrtf(var);
                x = __fadd_rn(mean, __fmul_rn(sd, eps));
            }
            nd[e] = x;
            // log_std = clip(log(sqrt(var)), -100, 1e8) (pens/utils.py:46-47); var = exp(2 log_std)
            float l = 0.5f * logvar, v2 = var;
            if (var == 0.f) { l = -100.f; v2 = 0.f; }                            // log(0) = -inf -> -100 -> exp(-200) = 0
            else if (isinf(var)) { l = 1e8f; }                                   // clip at 1e8 -> exp(2e8) = inf
            if (logvar != logvar) { l = logvar; v2 = logvar; }
            ls[e] = l; vr[e] = v2;
            rv[e] = FAST ? __fdividef(1.0f, __fadd_rn(v2, 1e-10f)) : __fdiv_rn(1.0f, __fadd_rn(v2, 1e-10f));
            if (e == member) sel = x;
        }
    }
    // np.var over the member axis (fake_env.py:112): sequential sums, true divides
    float s = 0.f;
#pragma unroll
    for (int e = 0; e < EMAX; ++e) if (e < E) s = (e == 0) ? nd[0] : __fadd_rn(s, nd[e]);
    const float m = FAST ? __fdividef(s, (float)E) : __fdiv_rn(s, (float)E);
    float q = 0.f;
#pragma unroll
    for (int e = 0; e < EMAX; ++e) if (e < E) {
        const float d = __fsub_rn(nd[e], m);
        const float d2 = __fmul_rn(d, d);
        q = (e == 0) ? d2 : __fadd_rn(q, d2);
    }
    EnvDimOut out;
    out.epv = FAST ? __fdividef(q, (float)E) : __fdiv_rn(q, (float)E);
    if (FAST) {
        // sum_{i,j} KL(N_i||N_j) without the O(E^2) loop: the log-std terms cancel and
        // sum_i (mu_j-mu_i)^2 = E d_j^2 + Q with d = mu - mean(mu), Q = sum d_i^2, so
        //   sum = 0.5 * sum_j (E d_j^2 + Q + sum_i var_i) / (var_j + 1e-10) - 0.5 E^2 .
        // Equal to the pairwise form up to float32 rounding (each pair is >= 0 analytically, so the
        // reference's per-pair clip at 0 only removes rounding noise); used by the throughput modes.
        float sv = 0.f;
#pragma unroll
        for (int e = 0; e < EMAX; ++e) if (e < E) sv += vr[e];
        const float qs = q + sv;
        float acc2 = 0.f;
#pragma unroll
        for (int e = 0; e < EMAX; ++e) if (e < E) {
            const float d = nd[e] - m;
            acc2 = fmaf(fmaf((float)E * d, d, qs), rv[e], acc2);
        }
        float tot = fmaf(0.5f, acc2, -0.5f * (float)(E * E));
        tot = (tot != tot) ? tot : fminf(fmaxf(tot, 0.0f), 1e10f * (float)(E * E));
        out.kl = __fdividef(tot, (float)((double)(E * (E - 1)) + 1e-10));
        out.nx = c.predicts_delta ? __fadd_rn(sel, obs_o) : sel;
        return out;
    }
    // average_dkl (pens/utils.py:30-57): all ordered pairs, i outer / j inner
    float acc = 0.f;
    bool first = true;
#pragma unroll
    for (int i = 0; i < EMAX; ++i) {
#pragma unroll
        for (int j = 0; j < EMAX; ++j) {
            if (i < E && j < E) {
                const float dm = __fsub_rn(nd[j], nd[i]);
                const float ratio = __fmul_rn(__fadd_rn(__fmul_rn(dm, dm), vr[i]), rv[j]);
                const float pre = __fsub_rn(__fadd_rn(__fmul_rn(0.5f, __fsub_rn(ratio, 1.0f)), ls[j]), ls[i]);
                const float k = (pre != pre) ? pre : fminf(fmaxf(pre, 0.0f), 1e10f);   // np.clip keeps nan
                acc = first ? k : __fadd_rn(acc, k);
                first = false;
            }
        }
    }
    out.kl = __fdiv_rn(acc, (float)((double)(E * (E - 1)) + 1e-10));             // pens/utils.py:56
    out.nx = c.predicts_delta ? __fadd_rn(sel, obs_o) : sel;                     // fake_env.py:125-131
    return out;
}

// row-owner part: ordered reductions over the O dimensions (numpy order), statics, reward
template <bool FAST, class Raw>
__device__ inline EnvRowOut env_row_finish(const EnvRowCfg& c, Raw raw, int member, const float* kl,
                                           const float* epv, const float* nx, const unsigned char* fin) {
    const int O = c.O;
    const float ks = np_sum(kl, O);
    const float es = np_sum(epv, O);
    bool all_finite = true;
    for (int o = 0; o < O; ++o) all_finite = all_finite && fin[o];
    // the next-state coordinates the statics read
    const float z = nx[0], q1 = O > 2 ? nx[2] : 0.f, q2 = O > 3 ? nx[3] : 0.f, last = nx[O - 1];
    EnvRowOut r;
    r.dkl_path = FAST ? __fdividef(ks, (float)O) : __fdiv_rn(ks, (float)O);      // fake_env.py:113
    r.ep_var_sum = es;
    r.ep_var_mean = FAST ? __fdividef(es, (float)O) : __fdiv_rn(es, (float)O);   // model_sampler.py:343
    auto notdone = [&]() {                                                       // statics.py:24-27
        const float zrot = __fsub_rn(1.0f, __fmul_rn(2.0f, __fadd_rn(__fmul_rn(q1, q1), __fmul_rn(q2, q2))));
        const bool flags = all_finite && (z >= 0.2f) && (z <= 1.0f);
        return __fmul_rn(flags ? 1.0f : 0.0f, zrot) >= -0.7f;
    };
    r.term = (c.term_id == CMBPO_TERM_ANTSAFE) ? !notdone() : false;             // statics.py:17-31
    if (c.cost_id == CMBPO_COST_HCS) {                                           // statics.py:10-15
        r.cost = (fabsf(__fmul_rn(last, 10.0f)) < 2.0f) ? 1.0f : 0.0f;
    } else if (c.cost_id == CMBPO_COST_ANTSAFE) {                                // statics.py:33-53
        const float cc = (!notdone() ? 1.0f : 0.0f) + ((fabsf(last) > 3.2f) ? 1.0f : 0.0f);
        r.cost = fminf(fmaxf(cc, 0.0f), 1.0f);
    } else {
        r.cost = 0.0f;                                                           // fake_env.py:146
    }
    int rcol = c.D - 1;
    if (c.predicts_cost) {                                                       // fake_env.py:139-142
        r.cost = __fadd_rn(__fmul_rn(c.sig_out[rcol], raw(member, rcol)), c.mu_out[rcol]);
        rcol -= 1;
    }
    r.rew = __fadd_rn(__fmul_rn(c.sig_out[rcol], raw(member, rcol)), c.mu_out[rcol]);   // :148-151
    return r;
}
