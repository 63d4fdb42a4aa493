"""`DeviceArchive`: the columns of the on-policy archive that start-state sampling reads
(`CPOBuffer.obs_archive`, `pi_info_archive['mu' / 'log_std']`, `epoch_archive`;
buffers/cpobuffer.py:110-137), resident on the GPU, with the sampling chain of
algorithms/cmbpo.py:241-245 on top:

    ep_b   = buffer.epoch_batch(B, buffer.epochs_list, ['observations', 'pi_infos'])   # cpobuffer.py:466
    kls    = clip(policy.compute_DKL(ep_b['observations'], ep_b['mu'], ep_b['log_std']), 0, None)
    dist   = buffer.boltz_dist(kls, alpha)                                             # cpobuffer.py:385
    btz_b  = buffer.distributed_batch_from_archive(B, dist, ['observations', 'pi_infos'])

`sample_start_states` runs all four on the device and returns the start states as a device tensor
that `ModelSampler.reset` accepts: no host<->device copy of observations per rollout batch.
Random draws come from Philox (seed, draw counter), not from numpy's global stream: equal in
distribution to the reference, reproducible for a seed.
"""
import ctypes as C

import numpy as np

from . import _lib as L


class DeviceArchive:
    def __init__(self, engine, archive_size, obs_dim, act_dim, seed=0):
        t = engine.torch
        self.engine, self.archive_size = engine, int(archive_size)
        self.obs_dim, self.act_dim = int(obs_dim), int(act_dim)
        self.observations = engine.zeros(self.archive_size, self.obs_dim)
        self.mu = engine.zeros(self.archive_size, self.act_dim)
        self.log_std = engine.zeros(self.archive_size, self.act_dim)
        self.epoch_archive = t.full((self.archive_size,), -1, dtype=t.int32, device=engine.device)
        self.archive_ptr = 0
        self.max_pointer = 0
        self.seed, self._draw = int(seed), 0
        self._index = None          # (sorted_idx, bin_offsets_dev, bin_offsets_host)

    # ---- filling (CPOBuffer.dump_to_archive, cpobuffer.py:209-247) ---------------------------
    def append(self, observations, mu, log_std, epochs):
        """Rows of one or more epochs, written at the ring pointer like dump_to_archive: when they
        do not fit (or fit exactly -- the reference's `>=`), the pointer wraps to 0 and the oldest rows are
        overwritten."""
        e, t = self.engine, self.engine.torch
        n = len(observations)
        assert n <= self.archive_size
        if self.archive_ptr >= self.archive_size - n:      # cpobuffer.py:221: an exact fit wraps too
            self.archive_ptr = 0
        sl = slice(self.archive_ptr, self.archive_ptr + n)
        self.observations[sl] = e.to_device(np.asarray(observations, np.float32), t.float32)
        self.mu[sl] = e.to_device(np.asarray(mu, np.float32), t.float32)
        self.log_std[sl] = e.to_device(np.asarray(log_std, np.float32), t.float32)
        self.epoch_archive[sl] = e.to_device(np.asarray(epochs, np.int32), t.int32)
        self.archive_ptr += n
        self.max_pointer = max(self.archive_ptr, self.max_pointer)
        self._index = None

    # ---- checkpoint and resume (checkpoint.save_state / load_state) ----------------------------
    def state_dict(self):
        """Rows [0, max_pointer) of the four columns (the rows past it were never written), the ring pointer, the seed
        and the draw counter that key the Philox draws."""
        n = self.max_pointer
        return {"precision": self.engine.precision_name, "archive_size": self.archive_size, "obs_dim": self.obs_dim,
                "act_dim": self.act_dim, "observations": self.observations[:n].cpu().numpy(),
                "mu": self.mu[:n].cpu().numpy(), "log_std": self.log_std[:n].cpu().numpy(),
                "epoch_archive": self.epoch_archive[:n].cpu().numpy(), "archive_ptr": self.archive_ptr,
                "max_pointer": n, "seed": self.seed, "draw": self._draw}

    @classmethod
    def from_state_dict(cls, engine, sd):
        """The inverse of state_dict(); the epoch index is rebuilt at the first draw."""
        engine.check_precision(sd["precision"])
        self = cls(engine, sd["archive_size"], sd["obs_dim"], sd["act_dim"], seed=sd["seed"])
        n, t = int(sd["max_pointer"]), engine.torch
        if not 0 <= int(sd["archive_ptr"]) <= n <= self.archive_size:
            raise ValueError("archive pointers %s / %s in an archive of %d rows"
                             % (sd["archive_ptr"], n, self.archive_size))
        for name, width in (("observations", self.obs_dim), ("mu", self.act_dim), ("log_std", self.act_dim),
                            ("epoch_archive", None)):
            shape = (n,) if width is None else (n, width)
            if tuple(sd[name].shape) != shape:
                raise ValueError("archive column %s is %s, want %s" % (name, tuple(sd[name].shape), shape))
            if n:
                getattr(self, name)[:n] = engine.to_device(sd[name], t.int32 if width is None else t.float32)
        self.archive_ptr, self.max_pointer, self._draw = int(sd["archive_ptr"]), n, int(sd["draw"])
        return self

    # ---- index by epoch ----------------------------------------------------------------------
    def _build_index(self):
        if self._index is not None:
            return self._index
        e, t = self.engine, self.engine.torch
        max_ep = int(self.epoch_archive.max().item())
        assert max_ep >= 0, "the archive is empty"
        n_bins = max_ep + 1
        sorted_idx = e.zeros(self.archive_size, dtype=t.int32)
        offs = e.zeros(n_bins + 1, dtype=t.int64)
        host = (C.c_int64 * (n_bins + 1))()
        L.check(e.lib.cmbpo_archive_index(e.h, e._p(self.epoch_archive), self.archive_size, n_bins,
                                          e._p(sorted_idx), e._p(offs), host))
        self._index = (sorted_idx, offs, np.frombuffer(host, dtype=np.int64).copy())
        return self._index

    @property
    def epoch_counts(self):
        """np.bincount(epoch_archive[epoch_archive >= 0]) (cpobuffer.py:151,392)."""
        return np.diff(self._build_index()[2])

    @property
    def epochs_list(self):
        """cpobuffer.py:149-154: the epochs that have rows, ascending."""
        return np.nonzero(self.epoch_counts)[0]

    @property
    def max_ep(self):
        return int(self.epochs_list[-1])

    @property
    def min_ep(self):
        return int(self.epochs_list[0])

    def _next_draw(self):
        self._draw += 1
        return self._draw

    # ---- epoch_batch + compute_DKL -------------------------------------------------------------
    def epoch_batch_indices(self, batch_size, epochs=None):
        """Row numbers [n_ep, batch_size] (device, int32): uniform rows of every epoch, with
        replacement -- `epoch_batch` (cpobuffer.py:515)."""
        e, t = self.engine, self.engine.torch
        sorted_idx, offs, _ = self._build_index()
        eps = self.epochs_list if epochs is None else np.asarray(epochs)
        eps_d = e.to_device(eps.astype(np.int32), t.int32)
        out = e.zeros(len(eps) * int(batch_size), dtype=t.int32)
        L.check(e.lib.cmbpo_archive_sample_epochs(e.h, e._p(sorted_idx), e._p(offs), e._p(eps_d), len(eps),
                                                  int(batch_size), self.seed, self._next_draw(), e._p(out)))
        return out.view(len(eps), int(batch_size))

    def gather(self, field, idx):
        e = self.engine
        src = getattr(self, field)
        flat = idx.reshape(-1)
        dst = e.empty(flat.numel(), src.shape[1])
        if flat.numel() == 0:                 # an empty shard: nothing to launch (and NULL pointers)
            return dst
        L.check(e.lib.cmbpo_gather_rows(e.h, e._p(src), src.shape[1], e._p(flat), flat.numel(), e._p(dst)))
        return dst

    def epoch_kls(self, policy, batch_size, epochs=None, precision=None):
        """`compute_DKL` of a 3-D epoch batch (cpo_policy.py:837-845): per epoch, the mean over
        batch_size sampled rows of KL(current policy || archived policy).  float64 [n_ep]."""
        e = self.engine
        idx = self.epoch_batch_indices(batch_size, epochs)
        n_ep = idx.shape[0]
        obs = self.gather("observations", idx)
        old_mu, old_ls = self.gather("mu", idx), self.gather("log_std", idx)
        cur_mu = e.policy_act(obs, eps=e.zeros(obs.shape[0], self.act_dim), precision=precision)["mu"]
        cur_ls = policy.log_std_device
        kl = (C.c_double * n_ep)()
        L.check(e.lib.cmbpo_policy_kl_epochs(e.h, e._p(cur_mu), e._p(cur_ls), e._p(old_mu), e._p(old_ls),
                                             n_ep, int(batch_size), self.act_dim, kl))
        return np.frombuffer(kl, dtype=np.float64).copy()

    # ---- boltz_dist (cpobuffer.py:385-396): host arithmetic on one number per epoch -------------
    def boltz_epoch_probs(self, kls, alpha=1):
        """Returns (ep_probs, sample_p): ep_probs[k] = probability of the k-th epoch of epochs_list,
        sample_p[e] = float32 probability of ONE row of epoch number e -- the two intermediate arrays
        of `boltz_dist`, computed with the same numpy operations."""
        ep_probs = np.exp(alpha * np.negative(kls))
        ep_probs /= np.sum(ep_probs)
        sample_p = self.epoch_counts.astype(np.float32)
        sample_p[sample_p > 0] = ep_probs / sample_p[sample_p > 0]
        return ep_probs, sample_p

    def boltz_dist(self, kls, alpha=1):
        """The reference's return value: per-ROW probabilities [archive_size] (numpy)."""
        _, sample_p = self.boltz_epoch_probs(kls, alpha)
        ep = self.epoch_archive.cpu().numpy()
        return np.where(ep >= 0, sample_p[ep], 0)

    # ---- distributed_batch_from_archive (cpobuffer.py:413-463) -----------------------------------
    def distributed_batch_indices(self, batch_size, kls, alpha=1, shard=None):
        """Row numbers [batch_size]: row r with probability boltz_dist(kls, alpha)[r].  `shard=(lo, hi)`:
        only entries lo:hi of that batch (the same draw counter advances either way)."""
        e, t = self.engine, self.engine.torch
        lo, hi = (0, int(batch_size)) if shard is None else (int(shard[0]), int(shard[1]))
        if not 0 <= lo <= hi <= int(batch_size):
            raise L.CmbpoError("shard %r is not inside a batch of %d" % (shard, batch_size))
        sorted_idx, offs, _ = self._build_index()
        eps = self.epochs_list
        _, sample_p = self.boltz_epoch_probs(kls, alpha)
        # the mass np.random.choice gives an epoch: (float32 row probability) x (rows), renormalised as
        # choice's cdf is (cdf /= cdf[-1])
        mass = sample_p[eps].astype(np.float64) * self.epoch_counts[eps]
        cdf = np.cumsum(mass)
        cdf /= cdf[-1]
        out = e.zeros(hi - lo, dtype=t.int32)
        eps_d = e.to_device(eps.astype(np.int32), t.int32)      # named: must outlive the launch
        cdf_d = e.to_device(cdf, t.float64)
        L.check(e.lib.cmbpo_archive_sample_boltz_range(e.h, e._p(sorted_idx), e._p(offs), e._p(eps_d), e._p(cdf_d),
                                                       len(eps), lo, hi - lo, self.seed, self._next_draw(),
                                                       e._p(out)))
        return out

    def sample_start_states(self, policy, batch_size, alpha=1, precision=None, shard=None, group=None):
        """algorithms/cmbpo.py:241-245 in one call.  Returns a dict of DEVICE tensors
        (observations [B,O], mu, log_std [B,A]) and the clipped per-epoch KLs (numpy).

        `shard=(lo, hi)`: rows lo:hi of what the call without `shard` returns (`batch_size` stays the
        whole batch).  Several ranks that hold the same archive and call this in step each get their block
        of one batch: every rank computes the per-epoch KLs, and when torch.distributed runs more than one
        rank in `group`, all of them use rank 0's (all-gathered), so that every rank draws from the same
        distribution bit for bit."""
        kls = np.clip(self.epoch_kls(policy, batch_size, precision=precision), a_min=0, a_max=None)
        if shard is not None:
            from .dist import all_gather_host, is_multi_rank
            if is_multi_rank(group):
                kls = all_gather_host(kls, group, self.engine.device)[0]
        idx = self.distributed_batch_indices(batch_size, kls, alpha, shard)
        return dict(observations=self.gather("observations", idx), mu=self.gather("mu", idx),
                    log_std=self.gather("log_std", idx), kls=kls, indices=idx)
