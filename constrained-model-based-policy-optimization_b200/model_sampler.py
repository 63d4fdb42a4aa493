"""`ModelSampler` with the reference's interface (samplers/model_sampler.py:12-444).

Two execution modes, same results:

* fused (policy is a `B200Policy` and env a `FakeEnv` of the same `Engine`): `reset()` launches
  the whole H-step rollout on the GPU speculatively -- paths are independent, noise is keyed by
  (global path id, step) -- and each `sample()` call just reveals one step and applies the two
  batch-global rules (max_samples cap, model_sampler.py:282-287; the caller's stop, cmbpo.py:258-263)
  as truncations of the finished rollout;
* step-wise (any policy object with get_action_outs/get_v/get_vc): the reference's control flow on
  the host, with env.step / buffer stores / GAE on the GPU.
"""
from collections import OrderedDict

import numpy as np

from . import _lib as L
from .dist import Ranks, cap_split, rank_order_sum
from .fake_env import FakeEnv
from .policy import B200Policy

EPS = 1e-8


class ModelSampler:
    def __init__(self, max_path_length, batch_size=1000, rollout_mode=False, logger=None,
                 seed=0):
        self._max_path_length = max_path_length
        self.batch_size = batch_size
        self.rollout_mode = rollout_mode
        self.logger = logger
        self.seed = int(seed)
        self._resets = 0
        self.env = self.policy = self.pool = None
        self.dkl_lim = None
        self._current_observation = None
        self._total_samples = 0
        self._total_dkl = 0
        self._n_episodes = 0
        self.injected = None          # tests: dict(act_eps=[T,B,A], elite_pos=[T,B], state_eps=...)
        self.path_id_base = 0         # multi-GPU: global id of this rank's first path
        self.return_arrays = False
        self._ranks = Ranks()         # the rollout block's ranks: this process alone until distribute()
        self._batch_total = batch_size
        self._global_sums = None

    # ---- plumbing identical to the reference ------------------------------------------------
    def initialize(self, env, policy, pool):
        self.env, self.policy, self.pool = env, policy, pool

    def set_policy(self, policy):
        self.policy = policy

    def set_logger(self, logger):
        self.logger = logger

    def terminate(self):
        self.env.close()

    def set_rollout_dkl(self, dkl):
        self.dkl_lim = dkl

    def set_max_path_length(self, path_length):
        self._max_path_length = path_length

    @property
    def dyn_dkl(self):
        return self._total_dkl / (self._total_samples + EPS)

    def batch_ready(self):
        return self.pool.size >= self.pool.max_size

    @property
    def fused(self):
        return (isinstance(self.policy, B200Policy) and isinstance(self.env, FakeEnv)
                and self.policy.engine is self.env.engine)

    # ---- multi-GPU ---------------------------------------------------------------------------
    def distribute(self, group=None, root=0):
        """Run the rollout block sharded over the ranks of `group` (torch.distributed, one process per
        GPU) with the samples one GPU gives.  Every rank calls reset() with its contiguous block of the
        start states, in rank order (DeviceArchive.sample_start_states(shard=...)).  The batch-wide
        rules -- the max_samples cap, the sample count and alive ratio the caller stops on,
        compute_dynamics_dkl and the finish_all_paths() diagnostics -- use counts and sums over all ranks
        and are identical on every rank, and the pool's get() returns the whole batch on rank `root` (zero
        rows elsewhere).  Without distribute() the same code runs with this process as the only rank.
        Fused mode only; call after initialize()."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()):
            raise L.CmbpoError("ModelSampler.distribute needs an initialised torch.distributed process group")
        if not self.fused:
            raise L.CmbpoError("a multi-rank ModelSampler needs the fused mode (a B200Policy and a FakeEnv of "
                               "one Engine); the step-wise mode runs on one rank only")
        self._ranks = Ranks.of(group, root)
        self._auto_base = self.path_id_base
        self.pool.distribute(group, root)

    # ---- checkpoint and resume (checkpoint.save_state / load_state) ----------------------------
    def state_dict(self):
        """The counters that key the rollouts' Philox draws (seed, resets, calibration calls) and the settings of the
        sampler.  Take it between batches: it raises while reset() has started a batch that get() has not returned.
        The sample and disagreement totals are kept too: compute_dynamics_dkl adds to them until the next reset().
        The ranks of distribute() are a runtime object and are not saved: call distribute() again after loading."""
        if self.pool is not None and self.pool.holds_batch:
            raise L.CmbpoError("a rollout batch is in flight: take the state after the pool's get()")
        return {"seed": self.seed, "resets": self._resets, "dkl_calls": getattr(self, "_dkl_calls", 0),
                "max_path_length": self._max_path_length,
                "dkl_lim": None if self.dkl_lim is None else float(self.dkl_lim), "batch_size": self.batch_size,
                "rollout_mode": self.rollout_mode, "total_samples": int(self._total_samples),
                "total_dkl": float(self._total_dkl)}

    @classmethod
    def from_state_dict(cls, sd):
        """The inverse of state_dict(); then initialize() (and distribute()) as for a new sampler."""
        self = cls(sd["max_path_length"], sd["batch_size"], sd["rollout_mode"], seed=sd["seed"])
        self._resets, self._dkl_calls = int(sd["resets"]), int(sd["dkl_calls"])
        self.dkl_lim = sd["dkl_lim"]
        self._total_samples, self._total_dkl = int(sd["total_samples"]), float(sd["total_dkl"])
        return self

    def _gather(self, vec):
        """[world, ...] all-gather of a small host vector, rank order."""
        return self._ranks.gather(vec, self.pool.engine.device)

    def _shard_base(self, n):
        """The global path count from the ranks' shard sizes.  After distribute(), also sets path_id_base (global
        id of this rank's first path); a single process keeps the caller's path_id_base."""
        sizes = self._gather(np.array([n], np.int64))[:, 0]
        if self._ranks.sharded:
            base = int(sizes[:self._ranks.rank].sum())
            if self.path_id_base not in (self._auto_base, base):
                raise L.CmbpoError("path_id_base %d was set by hand, but the shard sizes put this rank's first "
                                   "path at %d" % (self.path_id_base, base))
            self.path_id_base = self._auto_base = base
        return int(sizes.sum())

    # ---- calibration (model_sampler.py:151-167) ----------------------------------------------
    def compute_dynamics_dkl(self, obs_batch, depth=1):
        if self.fused:
            return self._dynamics_dkl_device(obs_batch, depth)
        self._require_fused_if_distributed()
        for _ in range(depth):
            outs = self.policy.get_action_outs(obs_batch)
            next_obs, _, terminal, info = self.env.step(obs_batch, outs["pi"])
            n_paths = next_obs.shape[0]
            self._total_dkl += info.get("ensemble_dkl_mean", 0) * n_paths
            self._total_samples += n_paths
            obs_batch = next_obs[np.squeeze(~terminal)]
        return self.dyn_dkl * depth

    def _dynamics_dkl_device(self, obs_batch, depth):
        """The same quantity from one `depth`-step device rollout that stores nothing (CMBPO_ROLLOUT_NO_STORE):
        step_stats[t] = (rows fed, sum of their disagreement, ..) so that
        sum_t mean_t * n_t = sum_t step_stats[t][1] and the sample count is sum_t step_stats[t][0]; rows of
        terminated paths leave the batch between steps as in the reference loop."""
        from .rollout import RolloutBuffers
        env = self.env
        eng = env.engine
        on_device = hasattr(obs_batch, "is_cuda") and obs_batch.is_cuda
        obs = obs_batch if on_device else np.asarray(obs_batch, np.float32)
        depth = int(depth)
        assert depth >= 1 and obs.shape[0] > 0
        bufs = RolloutBuffers(eng, obs.shape[0], depth + 1, env.obs_dim, env.act_dim, lean=True)
        inj = self.injected or {}
        bufs.set_inputs(obs, inj.get("act_eps"), inj.get("elite_pos"), inj.get("state_eps"))
        self._dkl_calls = getattr(self, "_dkl_calls", 0) + 1
        self._shard_base(obs.shape[0])    # obs_batch is this rank's block of the calibration batch
        bufs.run(env.env_cfg(True), uncertainty_mode=False, seed=(self.seed << 20) + (1 << 19) + self._dkl_calls,
                 path_id_base=self.path_id_base, max_steps=depth)
        st = self._step_stats(bufs, depth)
        self._total_dkl += float(st[:, 1].sum())
        self._total_samples += int(st[:, 0].sum())
        return self.dyn_dkl * depth

    # ---- reset (model_sampler.py:203-237) ----------------------------------------------------
    def _require_fused_if_distributed(self):
        if self._ranks.sharded and not self.fused:
            raise L.CmbpoError("a multi-rank ModelSampler runs the fused mode only: the step-wise mode "
                               "(external policy objects) runs on one rank")

    def reset(self, observations):
        """`observations`: the start states; after distribute(), this rank's contiguous block of them."""
        # a device tensor (DeviceArchive.sample_start_states) stays on the device in fused mode
        on_device = hasattr(observations, "is_cuda") and observations.is_cuda
        if not (on_device and self.fused):
            observations = np.asarray(observations.cpu() if on_device else observations, np.float32)
        self.batch_size = observations.shape[0]
        self._global_sums = None
        self._require_fused_if_distributed()
        self._batch_total = self._shard_base(self.batch_size)
        self._current_observation = observations
        self.policy.reset()
        self.pool.reset(self.batch_size)
        B = self.batch_size
        self._path_length = np.zeros(B)
        self._path_return = np.zeros(B)
        self._path_cost = np.zeros(B)
        self._path_dyn_var = np.zeros(B)
        self._dyn_dkl_path = np.zeros(B)
        self._total_samples = 0
        self._n_episodes = 0
        self._total_Vs = self._total_CVs = 0
        self._total_cost = self._total_rew = 0
        self._total_dyn_ep_var = 0
        self._total_dkl = 0
        self._max_dkl = 0
        self._max_path_return = 0
        self._resets += 1
        if self.fused:
            self._launch_fused(observations)

    # ---- fused mode ----------------------------------------------------------------------------
    def _launch_fused(self, observations):
        pool, env = self.pool, self.env
        bufs = pool.bufs
        inj = self.injected or {}
        bufs.set_inputs(observations, inj.get("act_eps"), inj.get("elite_pos"), inj.get("state_eps"))
        # a path ends once path_length >= max_path_length - 1 AFTER a store (model_sampler.py:352): the
        # reference stores max(1, H - 1) steps per path, also for H = 1 (schedule mode with min_length 1)
        steps = max(1, min(self._max_path_length, pool.max_path_length) - 1)
        bufs.run(env.env_cfg(True), uncertainty_mode=(self.rollout_mode == "uncertainty"),
                 dkl_lim=self.dkl_lim if self.dkl_lim is not None else 0.0,
                 seed=(self.seed << 20) + self._resets, path_id_base=self.path_id_base,
                 max_steps=steps)
        pool.adopt_device_rollout(self.policy.log_std)
        # the rollout is only queued: reset() returns immediately, the first sample() waits for it
        # (so a caller may prepare / finish another batch while this one runs)
        self._hist = None
        self._step_stats_host = None
        self._alive_now = self._batch_total
        self._stopped = False
        self._horizon_steps = steps

    def _counts(self, t):
        """(rows alive at the start of step t, of which cut as too uncertain at t, survivors)."""
        if self._hist is None:                      # first use after reset(): waits for the rollout
            self._hist = self._histogram()
            self._step_stats_host = self._step_stats(self.pool.bufs)
        h_len, h_unc = self._hist
        longer = int(h_len[t + 1:].sum())
        return longer + int(h_unc[t]), int(h_unc[t]), longer

    def _step_stats(self, bufs, steps=None):
        """(rows fed, sum of their disagreement) of each step (step_stats[:, 0:2]), summed over the ranks."""
        st = bufs.step_stats.cpu().numpy()[:steps]
        return rank_order_sum(self._gather(np.ascontiguousarray(st[:, 0:2])))

    def _histogram(self):
        """The length histograms of the batch (cmbpo_rollout_histogram), summed over the ranks, with the ranks'
        own length histograms kept in self._rank_h_len for the cap split."""
        h_len, h_unc = self.pool.bufs.histogram()
        g = self._gather(np.concatenate([h_len, h_unc]))
        self._rank_h_len = g[:, :len(h_len)]
        s = rank_order_sum(g)
        return s[:len(h_len)], s[len(h_len):]

    def _sample_fused(self, max_samples):
        t = self._n_episodes
        self._n_episodes += 1
        bufs = self.pool.bufs
        alive0, uncertain, survivors = self._counts(t)
        if max_samples:                                           # model_sampler.py:282-287
            n = max(self._total_samples + alive0 - uncertain - max_samples, 0)
            n = min(n, survivors)
            if n > 0:       # the first n survivors of the whole batch: this rank's share of them
                cut = cap_split(n, self._rank_h_len[:, t + 1:].sum(axis=1))[self._ranks.rank]
                if cut > 0:
                    bufs.truncate(cap_step=t, cap_n=cut)
                self._hist = self._histogram()
                survivors -= n
        self._total_samples += survivors
        self.pool.ptr = t + 1 if survivors > 0 else self.pool.ptr
        h_len, h_unc = self._hist
        # alive after the step: longer paths + paths that will be cut as uncertain next step
        alive_after = int(h_len[t + 2:].sum()) + (int(h_unc[t + 1]) if t + 1 < len(h_unc) else 0)
        if t + 1 >= self._horizon_steps:
            alive_after = 0
        self._alive_now = alive_after
        stats = self._step_stats_host[t]
        dkl_mean = stats[1] / stats[0] if stats[0] > 0 else 0.0
        info = {"ensemble_dkl_mean": np.float32(dkl_mean),
                "alive_ratio": alive_after / self._batch_total if survivors > 0 else 0}
        self._total_dkl += dkl_mean * survivors
        if self.return_arrays:
            m = (bufs.length > t)
            return (bufs.nextobs[t][m].cpu().numpy(), bufs.rew[t][m].cpu().numpy(),
                    bufs.term[t][m].cpu().numpy().astype(bool), info)
        return None, None, None, info

    def _finish_fused(self):
        bufs = self.pool.bufs
        if self._alive_now > 0:
            # close everything still alive after step n_episodes-1 (finish_all_paths, :418-444)
            bufs.truncate(stop_step=self._n_episodes - 1)
            self._alive_now = 0
        self.pool.finish_all_device()
        # one pass over the valid steps on the device (float64): the host accumulators of
        # model_sampler.py:314-333 and the sums of get_diagnostics (:89-133)
        B = bufs.B
        d = bufs.diagnostics()
        self._path_return = bufs.path_return.cpu().numpy()
        self._path_cost = bufs.path_cost.cpu().numpy()
        max_len = int(bufs.length.max().item()) if B else 0
        # sums over the ranks in rank order, maxima over the ranks: the same dict on every rank
        sums = ("rew", "cost", "val", "cval", "dyn_error", "n")
        v = np.array([d[k] for k in sums] + [self.pool.size, self._path_return.sum(), self._path_cost.sum(),
                                             d["max_dkl"], d["max_path_return"], max_len], np.float64)
        g = self._gather(v)
        s, m = rank_order_sum(g), g.max(axis=0)
        d.update(zip(sums, (float(x) for x in s[:6])))
        self._global_sums = (int(s[6]), float(s[7]), float(s[8]))
        d["max_dkl"], d["max_path_return"], max_len = float(m[9]), float(m[10]), int(m[11])
        self._total_rew, self._total_cost = d["rew"], d["cost"]
        self._total_Vs, self._total_CVs = d["val"], d["cval"]
        self._total_dyn_ep_var = d["dyn_error"] * bufs.O
        self._max_dkl = d["max_dkl"] if self._total_samples else 0
        self._max_path_return = max(0.0, d["max_path_return"]) if self._total_samples else 0
        self.pool.ptr = max_len

    # ---- sample (model_sampler.py:239-375) ---------------------------------------------------
    def sample(self, max_samples=None):
        assert self.pool.has_room
        assert self._current_observation is not None
        if self.fused:
            assert self._alive_now > 0
            return self._sample_fused(max_samples)
        self._require_fused_if_distributed()
        return self._sample_stepwise(max_samples)

    def _sample_stepwise(self, max_samples):
        pool = self.pool
        assert pool.alive_paths.any()
        self._n_episodes += 1
        alive = pool.alive_paths
        cur = self._current_observation
        outs = self.policy.get_action_outs(cur)
        a, logp, pi_info = outs["pi"], outs["logp_pi"], outs["pi_info"]
        v, vc = outs["v"], outs["vc"]
        nxt, rew, term, info = self.env.step(cur, a)
        rew = np.squeeze(rew, axis=-1)
        c = np.squeeze(info.get("cost", np.zeros(rew.shape)))
        term = np.squeeze(term, axis=-1)
        dkl_mean = info.get("ensemble_dkl_mean", 0)
        dkl_path = info.get("ensemble_dkl_path", 0)
        ep_var = info.get("ensemble_ep_var", np.zeros(shape=rew.shape[1:]))
        if self.rollout_mode == "uncertainty":
            cut = (self._dyn_dkl_path[alive] + dkl_path) >= self.dkl_lim
        else:
            cut = np.zeros(alive.sum(), dtype=bool)
        if max_samples:
            n = self._total_samples + alive.sum() - cut.sum()
            n = max(n - max_samples, 0)
            early = np.zeros((~cut).sum(), dtype=bool)
            early[:n] = True
            cut[~cut] = early
        keep = self._finish_paths(cut, True, True)
        alive = pool.alive_paths
        if not alive.any():
            info["alive_ratio"] = 0
            return nxt, rew, term, info
        cur, a, nxt, rew, v, c, vc, term, dkl_path, logp, ep_var = (
            x[keep] for x in (cur, a, nxt, rew, v, c, vc, term, dkl_path, logp, ep_var))
        pi_info = {k: x[keep] for k, x in pi_info.items()}
        n_alive = alive.sum()
        self._total_samples += n_alive
        self._total_cost += c.sum()
        self._total_rew += rew.sum()
        self._path_return[alive] += rew
        self._path_cost[alive] += c
        self._path_length[alive] += 1
        self._path_dyn_var[alive] += np.mean(ep_var, axis=-1)
        self._total_dyn_ep_var += ep_var.sum()
        self._total_Vs += v.sum()
        self._total_CVs += vc.sum()
        self._total_dkl += dkl_mean * n_alive
        self._max_dkl = max(self._max_dkl, np.max(dkl_path))
        self._dyn_dkl_path[alive] += dkl_path
        self._max_path_return = max(self._max_path_return, np.max(self._path_return))
        pool.store_multiple(cur, a, nxt, rew, v, c, vc, np.mean(ep_var, axis=-1), logp, pi_info, term)
        self._current_observation = nxt
        end = (self._path_length >= self._max_path_length - 1)[alive]
        keep = self._finish_paths(end, True, True)
        if not keep.any():
            info["alive_ratio"] = 0
            return nxt, rew, term, info
        self._current_observation = self._current_observation[keep]
        keep = self._finish_paths(term, False, True)
        if not keep.any():
            info["alive_ratio"] = 0
            return nxt, rew, term, info
        self._current_observation = self._current_observation[keep]
        info["alive_ratio"] = pool.alive_paths.sum() / self.batch_size
        return nxt, rew, term, info

    def _finish_paths(self, term_mask, append_vals=False, append_cvals=False):
        """model_sampler.py:377-416."""
        term_mask = np.asarray(term_mask, dtype=bool)
        if not term_mask.any():
            return np.logical_not(term_mask)
        obs = self._current_observation[term_mask]
        last_val = self.policy.get_v(obs) if append_vals else np.zeros(term_mask.sum())
        last_cval = self.policy.get_vc(obs) if append_cvals else np.zeros(term_mask.sum())
        self.pool.finish_path_multiple(term_mask, last_val, last_cval)
        return np.logical_not(term_mask)

    def finish_all_paths(self):
        """model_sampler.py:418-444."""
        if self.fused:
            self._finish_fused()
            return self.get_diagnostics()
        alive = self.pool.alive_paths
        if alive.any():
            mask = np.ones(alive.sum(), dtype=bool)
            self.pool.finish_path_multiple(mask, self.policy.get_v(self._current_observation),
                                           self.policy.get_vc(self._current_observation))
        assert self.pool.alive_paths.sum() == 0
        return self.get_diagnostics()

    def get_diagnostics(self):
        """model_sampler.py:89-133 (keys and formulas)."""
        n = self._total_samples + EPS
        if self._global_sums is None:
            size, ret_sum, cost_sum = self.pool.size, np.sum(self._path_return), np.sum(self._path_cost)
        else:
            size, ret_sum, cost_sum = self._global_sums
        d = OrderedDict({"pool-size": size})
        d.update({
            "msampler/samples_added": self._total_samples,
            "msampler/rollout_H_max": self._n_episodes,
            "msampler/rollout_H_mean": self._total_samples / (self._batch_total + EPS),
            "msampler/rew_var_perstep": 0 / n,
            "msampler/cost_var_perstep": 0 / n,
            "msampler/dyn_var_perstep": self._total_dyn_ep_var / n,
            "msampler/cost_rate": cost_sum / n,
            "msampler/rew_rate": ret_sum / n,
            "msampler/v_mean": self._total_Vs / n,
            "msampler/cv_mean": self._total_CVs / n,
            "msampler/ens_DKL": self._total_dkl / n,
            "msampler/ens_mean_var": 0 / n,
            "msampler/max_path_return": self._max_path_return,
            "msampler/max_dkl": self._max_dkl,
        })
        return d
