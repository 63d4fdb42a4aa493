/*
 * cmbpo_b200.h -- C ABI of libcmbpo_b200.so: the B200 (sm_100a) implementation of CMBPO's
 * model-rollout + GAE hot path.
 *
 * The reference (anyboby/Constrained-Model-Based-Policy-Optimization) has no FFI: its boundary
 * is three duck-typed Python interfaces.  Every entry point below names the reference
 * interface (file:line, relative to the reference root) whose arithmetic it replaces; the
 * Python classes in constrained-model-based-policy-optimization_b200/ keep the reference's
 * signatures and call these through ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; cmbpo_last_error() returns
 *     a thread-local message for the last failure;
 *   - all tensor pointers are DEVICE pointers (on the context's device) unless the name
 *     ends in _host; the caller owns them;
 *   - work is enqueued on the context's stream (cmbpo_ctx_set_stream) with no host
 *     synchronisation unless stated;
 *   - float = IEEE binary32; masks are uint8 (0/1); indices int32.
 *   - there is no CPU fallback: without a CUDA device cmbpo_ctx_create fails.
 */
#ifndef CMBPO_B200_H
#define CMBPO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CMBPO_ABI_VERSION 2

typedef struct cmbpo_ctx cmbpo_ctx;

/* which network a call addresses */
enum { CMBPO_NET_DYN = 0,   /* dynamics PE: models/pens/pe.py, built at algorithms/cmbpo.py:120-136 */
       CMBPO_NET_V = 1,     /* value ensemble:      policies/cpo_policy.py:467 */
       CMBPO_NET_VC = 2,    /* cost-value ensemble: policies/cpo_policy.py:468 */
       CMBPO_NET_ACTOR = 3, /* Gaussian actor mean MLP: network/ac_network.py:99-123 (E = 1) */
       CMBPO_NET_COUNT = 4 };

/* models/pens/fc.py:13-20 */
enum { CMBPO_ACT_NONE = 0, CMBPO_ACT_SWISH = 1, CMBPO_ACT_TANH = 2, CMBPO_ACT_RELU = 3,
       CMBPO_ACT_SIGMOID = 4 };

/* arithmetic of the GEMM chain */
enum { CMBPO_PREC_FP32 = 0,   /* CUDA-core fp32: the variant that isolates logic from precision */
       CMBPO_PREC_BF16 = 1,   /* tcgen05 kind::f16, bf16 operands, fp32 accumulate in TMEM */
       CMBPO_PREC_FP16 = 2,   /* tcgen05 kind::f16, fp16 operands (tf32-class mantissa), fp32 accumulate */
       CMBPO_PREC_BF16_X2 = 3, /* reserved (removed: packed 16-bit activation arithmetic gained nothing -- */
       CMBPO_PREC_FP16_X2 = 4 }; /* the MUFU rate is per element); passing them is an error */

/* models/statics.py:56-70 */
enum { CMBPO_TERM_NO_DONE = 0, CMBPO_TERM_ANTSAFE = 1 };
enum { CMBPO_COST_ZERO = 0, CMBPO_COST_HCS = 1, CMBPO_COST_ANTSAFE = 2 };

/* why a model path ended (samplers/model_sampler.py:275-367, 418-444) */
enum { CMBPO_END_ALIVE = 0, CMBPO_END_UNCERTAIN = 1, CMBPO_END_HORIZON = 2, CMBPO_END_TERMINAL = 3,
       CMBPO_END_CAPPED = 4,  /* max_samples cap, model_sampler.py:282-287 */
       CMBPO_END_STOPPED = 5  /* finish_all_paths after the caller stopped, model_sampler.py:418-444 */ };

/* GAE scan flavour */
enum { CMBPO_SCAN_STRICT = 0, /* float64, strictly sequential: bit-identical to scipy.signal.lfilter */
       CMBPO_SCAN_WARP = 1 }; /* float64 warp-shuffle segmented scan (re-associated; <= 1 ulp after the fp32 round) */

int cmbpo_abi_version(void);
const char* cmbpo_last_error(void);

int cmbpo_ctx_create(int device, cmbpo_ctx** out);
int cmbpo_ctx_destroy(cmbpo_ctx* ctx);
int cmbpo_ctx_set_stream(cmbpo_ctx* ctx, void* cuda_stream);
int cmbpo_ctx_synchronize(cmbpo_ctx* ctx);
/* number of this library's kernels launched on the context since creation (bench.py's gpu_launches) */
int64_t cmbpo_ctx_launch_count(cmbpo_ctx* ctx);
/*
 * Measurement hooks (bench.py's roofline): when enabled, CUDA events are recorded on the
 * context's stream around every launch of the dominant kernels.  slot 0 = the dynamics-ensemble
 * GEMM chain (K1), slot 1 = the GAE scan (K3), slot 2 = the rollout row kernel (K2), slot 3 = the
 * policy pass (actor + V + VC chains + row kernel).  _read synchronises, returns the summed device
 * time and the number of bracketed launches, and optionally resets the slot.
 */
enum { CMBPO_PROF_DYN = 0, CMBPO_PROF_GAE = 1, CMBPO_PROF_STEP = 2, CMBPO_PROF_POLICY = 3, CMBPO_PROF_SLOTS = 4 };
int cmbpo_ctx_profile(cmbpo_ctx* ctx, int enable);
int cmbpo_ctx_profile_read(cmbpo_ctx* ctx, int slot, double* total_ms_host, int64_t* launches_host,
                           int reset);

/*
 * Upload one network.  Replaces the TF variables behind models/pens/fc.py:123-170 (weights
 * [E,in,out], biases [E,1,out]) and models/pens/utils.py:104-111 (scaler mu/var [1,dim]).
 *   dims[n_layers+1], W[l] -> [E, dims[l], dims[l+1]], b[l] -> [E, dims[l+1]], acts[n_layers].
 *   For a probabilistic net dims[n_layers] = 2*D (mean | logvar), models/pens/pe.py:179-180.
 *   mu_* / var_* may be NULL (no scaler).  elite_inds: models/pens/pe.py:396-403 (may hold duplicates).
 *   on_device != 0: the arrays are already on the device (e.g. after an NCCL broadcast).
 */
int cmbpo_net_set_weights(cmbpo_ctx* ctx, int which, int E, int n_layers, const int* dims_host,
                          const float* const* W, const float* const* b, const int* acts_host,
                          const float* mu_in, const float* var_in, const float* mu_out,
                          const float* var_out, int probabilistic, const int* elite_inds_host,
                          int n_elite, int on_device);
/* state-independent log_std of the actor, network/ac_network.py:104 */
int cmbpo_actor_set_log_std(cmbpo_ctx* ctx, const float* log_std, int A, int on_device);

/*
 * PE.predict_ensemble (models/pens/pe.py:671-713 -> _compile_outputs 789-838).
 *   x: [N, in] (x_is_3d = 0, fc.py:87-88) or [E, N, in] (x_is_3d = 1, fc.py:89-90).
 *   mean, var: [E, N, D]; var may be NULL for a non-probabilistic net.
 */
int cmbpo_ens_predict(cmbpo_ctx* ctx, int which, const float* x, int64_t N, int x_is_3d,
                      float* mean, float* var, int precision);
/* PE.predict (pe.py:648-669, tensors 326-330 / 343): mean over ALL members -> [N, D]; var may be NULL */
int cmbpo_ens_predict_mean(cmbpo_ctx* ctx, int which, const float* x, int64_t N, float* mean,
                           float* var, int precision);

/*
 * CPOPolicy.get_action_outs (policies/cpo_policy.py:801-823; ac_network.py:99-123, 46-48).
 *   eps: [N, A] injected standard normals, or NULL -> Philox4x32-10 keyed (seed, path id, step).
 *   path_ids: [N] global path id per row (NULL -> row index).  Outputs: pi, mu [N,A]; logp, v, vc [N].
 */
int cmbpo_policy_act(cmbpo_ctx* ctx, const float* obs, int64_t N, const float* eps,
                     const int32_t* path_ids, uint64_t seed, int step, float* pi, float* logp,
                     float* mu, float* v, float* vc, int precision);

/*
 * FakeEnv.step for 2-D inputs (models/fake_env.py:66-172) with an ensemble, probabilistic,
 * delta-predicting model that also predicts the reward (algorithms/cmbpo.py:137-142).
 *   elite_pos: [N] positions into elite_inds (what np.random.choice draws, fake_env.py:174-176)
 *              or NULL -> Philox.   state_eps: [N,O] multiplier of std when deterministic = 0
 *              (NULL -> 1, the reference's `+ std`, fake_env.py:105-106).
 *   next_obs [N,O], rew [N], cost [N], term [N] u8, dkl_path [N], ep_var [N,O],
 *   dkl_mean_out: 1 float (ensemble_dkl_mean).
 */
typedef struct {
    int term_id, cost_id;      /* models/statics.py tables */
    int predicts_cost;         /* fake_env.py:139-142 */
    int deterministic;         /* fake_env.py:105-108 */
    int predicts_delta;        /* fake_env.py:130-131 */
} cmbpo_env_cfg;

int cmbpo_fakeenv_step(cmbpo_ctx* ctx, const cmbpo_env_cfg* cfg, const float* obs, const float* act,
                       int64_t N, const int32_t* elite_pos, const float* state_eps,
                       const int32_t* path_ids, uint64_t seed, int step, float* next_obs, float* rew,
                       float* cost, uint8_t* term, float* dkl_path, float* ep_var,
                       float* dkl_mean_out, int precision);

/*
 * The H-step model rollout: ModelSampler.reset + sample x (T-1) (samplers/model_sampler.py:203-375)
 * writing what ModelBuffer.store_multiple would (buffers/modelbuffer.py:114-135), for B start
 * states.  Per-path rules (uncertainty cut-off, horizon, env terminal) are applied in the
 * kernel; the two batch-global rules (max_samples cap, alive-ratio stop) are a truncation
 * applied afterwards by cmbpo_rollout_truncate.
 *
 * Buffers are TIME-MAJOR: field[t][p][...] with t < T = max_path_length, p < B, so that one
 * step of 128 consecutive paths is one contiguous, coalesced block.
 */
typedef struct {
    /* inputs */
    const float* start_obs;      /* [B,O] */
    const float* act_eps;        /* [T,B,A] or NULL (Philox) */
    const int32_t* elite_pos;    /* [T,B]   or NULL (Philox) */
    const float* state_eps;      /* [T,B,O] or NULL */
    /* per-step fields, time-major */
    float *obs, *act, *nextobs, *mu;               /* [T,B,O], [T,B,A], [T,B,O], [T,B,A] */
    float *rew, *val, *cost, *cval, *logp, *dyn_error, *dkl; /* [T,B] */
    uint8_t* term;                                 /* [T,B] */
    /* per-path results */
    int32_t* length;             /* [B] stored steps */
    uint8_t* end_reason;         /* [B] CMBPO_END_* */
    float *last_val, *last_cval; /* [B] bootstrap values for the GAE pass */
    double *cum_dkl, *path_return, *path_cost; /* [B] float64 accumulators, model_sampler.py:218-226 */
    float* final_obs;            /* [B,O] current observation of every path still alive at the end */
    double* step_stats;          /* [T,4] per step: rows fed to the model, sum of dkl_path over them,
                                    rows stored, sum of ensemble_ep_var over the stored rows */
} cmbpo_rollout_bufs;

typedef struct {
    int64_t B;                   /* start states on this rank */
    int64_t path_id_base;        /* global id of path 0 (multi-GPU shard offset; keys the Philox streams) */
    int T;                       /* max_path_length (maxroll); at most T-1 steps are stored, model_sampler.py:352 */
    int max_steps;               /* stop after this many steps (<= T-1), <=0 -> T-1 */
    int uncertainty_mode;        /* rollout_mode == 'uncertainty', model_sampler.py:275 */
    double dkl_lim;              /* model_sampler.py:171-172 */
    uint64_t seed;
    int precision;
    cmbpo_env_cfg env;
    int flags;                   /* CMBPO_ROLLOUT_* bits (ABI 2) */
    int compact_every;           /* steps between alive-row compactions; <= 0 -> 2 (ABI 2) */
} cmbpo_rollout_cfg;

/* cmbpo_rollout_cfg.flags.  None of them changes a result bit (tests compare both settings):
 *   NO_COMPACT  keep finished paths' rows in the batch (see below);
 *   FUSE        tensor-core precisions: run the step as TWO launches -- the policy GEMM, and the dynamics
 *               GEMM kernel with the policy head in its input staging and the FakeEnv row math / sampler
 *               rules / ModelBuffer write-out in its epilogue (raw outputs only tile by tile in an
 *               L2-resident scratch) -- instead of the default four (policy GEMM, policy rows, dynamics
 *               GEMM with raw [E,B,2D] outputs in HBM, row kernel).  Bit-identical; opt-in because it is
 *               currently slower (the row math occupies the GEMM kernel's epilogue warps);
 *   NO_STORE    do not write the per-step ModelBuffer fields (obs .. term may then be NULL): only the
 *               per-path results and step_stats -- ModelSampler.compute_dynamics_dkl
 *               (samplers/model_sampler.py:151-167) = sum_t step_stats[t][1] / sum_t step_stats[t][0]. */
enum { CMBPO_ROLLOUT_NO_COMPACT = 1, CMBPO_ROLLOUT_FUSE = 2, CMBPO_ROLLOUT_NO_STORE = 4 };

/* Like the reference (model_sampler.py:255-259, 300-311) only alive paths are fed to the networks: on
 * the tensor-core precisions, where paths can end early (termination function / uncertainty mode), the
 * rows of finished paths are compacted out of the batch on the device every other step; results do
 * not depend on it (bit-identical).  final_obs is written for the paths still alive at the end.
 * Host synchronisation: none without compaction.  With compaction the live row count is mirrored to the
 * host after every compaction and the call waits (cudaEventSynchronize) for the count of the compaction
 * THREE back before issuing further steps, so that it can stop once no path is alive; the call therefore
 * returns at most 3 compactions ahead of the device. */
int cmbpo_rollout(cmbpo_ctx* ctx, const cmbpo_rollout_cfg* cfg, const cmbpo_rollout_bufs* bufs);

/*
 * Batch-global rules of the sampler, applied to a finished speculative rollout as a truncation
 * (paths are independent, so cutting path p at step t only shortens it):
 *   - max_samples cap (model_sampler.py:282-287): at step cap_step the first cap_n surviving paths
 *     BY PATH INDEX are closed before the step is stored, bootstrapped with V(s_t), VC(s_t);
 *   - stop (algorithms/cmbpo.py:258-263 then model_sampler.py:418-444 finish_all_paths): after step
 *     stop_step every path still alive is closed, bootstrapped with V(s_{t+1}), VC(s_{t+1}).
 * The host decides cap_step / cap_n / stop_step from the histogram (host-synchronous, 2*(T+1)
 * int64: count(length == L) and count(length == L and end_reason == UNCERTAIN)).
 * Pass cap_step < 0 / stop_step < 0 to skip a rule.
 */
int cmbpo_rollout_histogram(cmbpo_ctx* ctx, const int32_t* length, const uint8_t* end_reason,
                            int64_t B, int T, int64_t* hist_host);
int cmbpo_rollout_truncate(cmbpo_ctx* ctx, const cmbpo_rollout_bufs* bufs, int64_t B, int T,
                           int cap_step, int64_t cap_n, int stop_step);

/*
 * Diagnostics of a finished (and truncated) rollout over the valid steps t < length[p], replacing the
 * per-step host accumulators of ModelSampler.sample (samplers/model_sampler.py:314-333) and the
 * sums of get_diagnostics (model_sampler.py:89-133).  path_return / path_cost: device [B] float64.
 * stats_host[8] (host, float64): sum rew, sum cost, sum val, sum cval, sum dyn_error, max dkl,
 * max running path return, number of steps.  Synchronises the stream.
 */
int cmbpo_rollout_diagnostics(cmbpo_ctx* ctx, const cmbpo_rollout_bufs* bufs, int64_t B,
                              double* path_return, double* path_cost, double* stats_host);

/*
 * Start-state sampling from the on-policy archive (algorithms/cmbpo.py:241-245), archive columns
 * resident on the device.  Randomness: Philox4x32-10 keyed (seed, draw, sample index).
 *
 * cmbpo_archive_index: stable counting sort of the rows by epoch (CPOBuffer.epoch_archive,
 *   buffers/cpobuffer.py:135,242; rows with epoch < 0 are empty).  sorted_idx [N] int32: row numbers
 *   grouped by epoch, ascending inside an epoch; bin_offsets [n_bins + 1] int64 (device) and its host
 *   copy: rows of epoch e are sorted_idx[bin_offsets[e] : bin_offsets[e + 1]].  Synchronises.
 * cmbpo_archive_sample_epochs: CPOBuffer.epoch_batch (cpobuffer.py:466-524):
 *   out_idx[k * B + b] = a uniform row of epoch epochs[k].
 * cmbpo_archive_sample_boltz: distributed_batch_from_archive with a boltz_dist distribution
 *   (cpobuffer.py:385-396, 413-463): epoch k with probability cdf[k] - cdf[k-1] (cdf [n_ep] float64,
 *   device), then a uniform row of it == np.random.choice(N, B, p=dist) in distribution.
 * cmbpo_gather_rows: dst[i, :] = src[idx[i], :]   (arch_dict[field][indices]).
 * cmbpo_policy_kl_epochs: CPOPolicy.compute_DKL for a 3-D batch (cpo_policy.py:837-845,
 *   network/ac_network.py:50-55): kl_host[k] = mean_b sum_a KL(current || archived) over the B rows of
 *   epoch slot k; cur_mu / old_mu / old_log_std [n_ep * B, A], cur_log_std [A].  Synchronises.
 */
int cmbpo_archive_index(cmbpo_ctx* ctx, const int32_t* epoch, int64_t N, int n_bins,
                        int32_t* sorted_idx, int64_t* bin_offsets, int64_t* bin_offsets_host);
int cmbpo_archive_sample_epochs(cmbpo_ctx* ctx, const int32_t* sorted_idx, const int64_t* bin_offsets,
                                const int32_t* epochs, int n_ep, int64_t B, uint64_t seed, uint64_t draw,
                                int32_t* out_idx);
int cmbpo_archive_sample_boltz(cmbpo_ctx* ctx, const int32_t* sorted_idx, const int64_t* bin_offsets,
                               const int32_t* epochs, const double* cdf, int n_ep, int64_t B,
                               uint64_t seed, uint64_t draw, int32_t* out_idx);
int cmbpo_gather_rows(cmbpo_ctx* ctx, const float* src, int width, const int32_t* idx, int64_t n, float* dst);
int cmbpo_policy_kl_epochs(cmbpo_ctx* ctx, const float* cur_mu, const float* cur_log_std, const float* old_mu,
                           const float* old_log_std, int n_ep, int64_t B, int A, double* kl_host);

/*
 * GAE + cost-GAE + returns over finished paths
 * (buffers/modelbuffer.py:163-179, buffers/cpobuffer.py:179-207, utilities/utils.py:159-211).
 *   element (p, t) of every field lives at p*path_stride + t*time_stride (in floats).
 *   length[p] steps are valid; last_val/last_cval [n_paths].  Writes adv, ret, cadv, cret for
 *   t < length[p] only.
 */
int cmbpo_gae_paths(cmbpo_ctx* ctx, const float* rew, const float* val, const float* cost,
                    const float* cval, int64_t n_paths, int max_len, int64_t path_stride,
                    int64_t time_stride, const int32_t* length, const float* last_val,
                    const float* last_cval, double gamma, double lam, double cgamma, double clam,
                    float* adv, float* ret, float* cadv, float* cret, int scan_mode);
/* flat CPOBuffer layout: segment i = [seg_offsets[i], seg_offsets[i+1]) (cpobuffer.py:180, 206) */
int cmbpo_gae_flat(cmbpo_ctx* ctx, const float* rew, const float* val, const float* cost,
                   const float* cval, int64_t n, const int64_t* seg_offsets, int64_t n_seg,
                   const float* last_val, const float* last_cval, double gamma, double lam,
                   double cgamma, double clam, float* adv, float* ret, float* cadv, float* cret,
                   int scan_mode);

/*
 * mpi_statistics_scalar (utilities/mpi_tools.py:71-92) pass 1 and 2 over the valid entries
 * (valid = t < length[p] for the path layout; all n for the flat layout when length == NULL).
 *   sums_out (device, 8 doubles): {n, sum_adv, sum_cadv, sum_ret, sum_cret, sumsq_adv(after pass 2), 0, 0}.
 *   Multi-GPU: the caller all-reduces sums_out[0..4] between pass 1 and pass 2 and sums_out[5]
 *   after pass 2 (the two Allreduce calls of mpi_tools.py:82-86).
 */
int cmbpo_adv_stats_pass1(cmbpo_ctx* ctx, const float* adv, const float* cadv, const float* ret,
                          const float* cret, int64_t n_paths, int max_len, int64_t path_stride,
                          int64_t time_stride, const int32_t* length, double* sums_out);
int cmbpo_adv_stats_pass2(cmbpo_ctx* ctx, const float* adv, int64_t n_paths, int max_len,
                          int64_t path_stride, int64_t time_stride, const int32_t* length,
                          float adv_mean, double* sums_out);
/* adv <- (adv-mean)/(std+1e-8), cadv <- cadv-cmean on valid entries (modelbuffer.py:198-204) */
int cmbpo_adv_normalise(cmbpo_ctx* ctx, float* adv, float* cadv, int64_t n_paths, int max_len,
                        int64_t path_stride, int64_t time_stride, const int32_t* length,
                        float adv_mean, float adv_std, float cadv_mean);
/*
 * The same two steps with the statistics kept in DEVICE memory (no host round trip between the passes, so a
 * multi-GPU job's ranks are only coupled by the two NCCL all-reduces, not by host synchronisations):
 * sums_dev = the 8 doubles of pass 1 (all-reduced); pass2_dev forms mean = float32(sum)/float32(n) on the device
 * (mpi_tools.py:82-83) and writes the local sum of squares to sums_out[5]; normalise_dev forms mean, cmean and
 * std = sqrt(float32(sumsq)/float32(n)) from the (all-reduced) sums (mpi_tools.py:85-86).  n == 0: no-ops.
 */
int cmbpo_adv_stats_pass2_dev(cmbpo_ctx* ctx, const float* adv, int64_t n_paths, int max_len,
                              int64_t path_stride, int64_t time_stride, const int32_t* length,
                              const double* sums_dev, double* sums_out);
int cmbpo_adv_normalise_dev(cmbpo_ctx* ctx, float* adv, float* cadv, int64_t n_paths, int max_len,
                            int64_t path_stride, int64_t time_stride, const int32_t* length,
                            const double* sums_dev);

/*
 * SURVEY.md 8f-4: the ensemble training step -- the body of the batch loop of PE.train (models/pens/pe.py:547-567).
 *   train_begin  allocates the optimiser state of slot `which` (Adam moments, zero; step counter 0).  The state
 *                persists across calls like tf.train.AdamOptimizer's variables; cmbpo_net_set_weights drops it.
 *   train_step   x [E,bs,in], y [E,bs,D] (device): member e trains on ITS OWN batch (bootstrap rows, pe.py:523,549).
 *                Forward (fc.py:74-95), loss, backward, Adam update of the fp32 master weights in place.
 *                loss = CMBPO_LOSS_MSPE (probabilistic nets; pe.py:921-973) or CMBPO_LOSS_MSE (pe.py:840-919 with
 *                inc_var_loss=False); weight_decay[l] multiplies tf.nn.l2_loss(W_l) (fc.py:168-169;
 *                pe_factory.py:50-55: decay/4, decay/2 ..., decay).  loss_out (device, [E], may be NULL): the
 *                per-member loss vector the reference's loss function returns (before decay).
 *                math: 0 = fp32 GEMMs, 1 = TF32 tensor-core GEMMs (cuBLAS).
 *   train_loss   `self.loss` of the reference (pe.py:264): mean 0.5 (mean - transform(y))^2 per member, no update.
 *   train_grads  device copies of the last step's gradients of one layer (before decay): dW [E,in,out], db [E,out].
 *   train_end    installs new elites (NULL keeps them) and re-packs the tcgen05 weight streams: predictions and
 *                rollouts after it see the trained weights (pe.py:396-399, 601-607).
 *   cmbpo_net_get_weights / cmbpo_net_set_scalers: device copies of one layer's variables; new scaler statistics
 *                (TensorStandardScaler.fit, pens/utils.py:119-138; host pointers).
 */
enum { CMBPO_LOSS_MSPE = 0, CMBPO_LOSS_MSE = 1 };
typedef struct {
    int loss;
    float lr, beta1, beta2, eps;       /* tf.train.AdamOptimizer: 1e-3 (cmbpo.py:51), 0.9, 0.999, 1e-8 */
    float weight_decay[8];
    int math;
} cmbpo_train_cfg;
int cmbpo_ens_train_begin(cmbpo_ctx* ctx, int which);
int cmbpo_ens_train_step(cmbpo_ctx* ctx, int which, const float* x, const float* y, int64_t bs,
                         const cmbpo_train_cfg* cfg, float* loss_out);
int cmbpo_ens_train_loss(cmbpo_ctx* ctx, int which, const float* x, const float* y, int64_t bs, float* loss_out);
int cmbpo_ens_train_grads(cmbpo_ctx* ctx, int which, int layer, float* dW, float* db);
int cmbpo_ens_train_end(cmbpo_ctx* ctx, int which, const int* elite_inds, int n_elite);
int cmbpo_net_get_weights(cmbpo_ctx* ctx, int which, int layer, float* W, float* b);
int cmbpo_net_set_scalers(cmbpo_ctx* ctx, int which, const float* mu_in, const float* var_in,
                          const float* mu_out, const float* var_out);

/*
 * ModelBuffer.get()'s `buf[populated_mask]` (modelbuffer.py:218): gathers the valid (p,t)
 * entries of a time-major field [T,B,width] into out[row,width], rows ordered path-major then
 * time (numpy boolean-mask order).  row_offsets [B+1] = exclusive prefix sum of length
 * (cmbpo_path_offsets).
 */
int cmbpo_path_offsets(cmbpo_ctx* ctx, const int32_t* length, int64_t B, int64_t* row_offsets);
int cmbpo_compact_field(cmbpo_ctx* ctx, const float* field, int64_t B, int T, int width,
                        const int32_t* length, const int64_t* row_offsets, float* out);

/*
 * ModelBuffer.store_multiple (modelbuffer.py:114-135) for callers that step an external policy:
 * dst is a time-major field [T,B,width]; row i of src [n,width] goes to path path_idx[i], column t.
 */
int cmbpo_scatter_rows(cmbpo_ctx* ctx, float* dst, int64_t B, int width, int t,
                       const int32_t* path_idx, const float* src, int64_t n);

#ifdef __cplusplus
}
#endif
#endif /* CMBPO_B200_H */
