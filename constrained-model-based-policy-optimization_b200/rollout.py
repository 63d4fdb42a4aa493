"""Device-side storage of one rollout batch and the thin wrappers over cmbpo_rollout /
cmbpo_rollout_truncate / cmbpo_gae_paths.

Layout (DESIGN.md "Data layout in HBM"): every per-step field is TIME-MAJOR, field[t][p][...],
t < T = max_path_length, p < B, so that step t of 128 consecutive paths is one contiguous block
(coalesced write-out from the rollout kernel, coalesced reads in the GAE scan).  The
reference's [B, T, ...] arrays (buffers/modelbuffer.py:53-98) are views produced on demand.
"""
import ctypes as C

import numpy as np

from . import _lib as L

STEP_FIELDS_VEC = ("obs", "act", "nextobs", "mu")
STEP_FIELDS = ("rew", "val", "cost", "cval", "logp", "dyn_error", "dkl")
GAE_FIELDS = ("adv", "ret", "cadv", "cret")


class RolloutBuffers:
    def __init__(self, engine, B, T, obs_dim, act_dim, lean=False):
        """`lean`: only the per-path results and the per-step statistics (for CMBPO_ROLLOUT_NO_STORE runs:
        the per-step ModelBuffer fields stay NULL)."""
        t = engine.torch
        self.engine, self.B, self.T, self.O, self.A = engine, int(B), int(T), int(obs_dim), int(act_dim)
        self.lean = bool(lean)
        z = engine.zeros
        if not lean:
            self.obs, self.nextobs = z(T, B, obs_dim), z(T, B, obs_dim)
            self.act, self.mu = z(T, B, act_dim), z(T, B, act_dim)
            for k in STEP_FIELDS + GAE_FIELDS:
                setattr(self, k, z(T, B))
            self.term = z(T, B, dtype=t.uint8)
        self.length = z(B, dtype=t.int32)
        self.end_reason = z(B, dtype=t.uint8)
        self.last_val, self.last_cval = z(B), z(B)
        self.cum_dkl, self.path_return, self.path_cost = (z(B, dtype=t.float64) for _ in range(3))
        self.final_obs = z(B, obs_dim)
        self.step_stats = z(T, 4, dtype=t.float64)
        self.start_obs = None
        self.act_eps = self.elite_pos = self.state_eps = None

    def struct(self):
        e = self.engine
        s = L.RolloutBufs()
        for name, _ in L.RolloutBufs._fields_:
            tns = getattr(self, name, None)
            setattr(s, name, None if tns is None else tns.data_ptr())
        # keep dtype discipline explicit
        assert self.length.dtype == e.torch.int32 and (self.lean or self.term.dtype == e.torch.uint8)
        return s

    def set_inputs(self, start_obs, act_eps=None, elite_pos=None, state_eps=None):
        e, t = self.engine, self.engine.torch
        self.start_obs = e.to_device(start_obs, t.float32)
        assert tuple(self.start_obs.shape) == (self.B, self.O)
        self.act_eps = None if act_eps is None else e.to_device(act_eps, t.float32)
        self.elite_pos = None if elite_pos is None else e.to_device(elite_pos, t.int32)
        self.state_eps = None if state_eps is None else e.to_device(state_eps, t.float32)
        if self.act_eps is not None:
            assert tuple(self.act_eps.shape[1:]) == (self.B, self.A) and self.act_eps.shape[0] >= self.T - 1
        if self.elite_pos is not None:
            assert self.elite_pos.shape[1] == self.B and self.elite_pos.shape[0] >= self.T - 1

    def run(self, env_cfg, uncertainty_mode=False, dkl_lim=0.0, seed=0, path_id_base=0,
            max_steps=0, precision=None, flags=0, compact_every=0):
        """cmbpo_rollout: the speculative per-path rollout.  `flags`: L.ROLLOUT_* bits (results do not
        depend on NO_COMPACT; FUSE is retired and ignored; NO_STORE leaves the per-step fields untouched)."""
        e = self.engine
        if self.lean:
            flags = int(flags) | L.ROLLOUT_NO_STORE
        cfg = L.RolloutCfg(self.B, int(path_id_base), self.T, int(max_steps),
                           int(bool(uncertainty_mode)), float(dkl_lim if dkl_lim is not None else 0.0),
                           int(seed), e._prec(precision), env_cfg, int(flags), int(compact_every))
        bufs = self.struct()
        L.check(e.lib.cmbpo_rollout(e.h, C.byref(cfg), C.byref(bufs)))

    def histogram(self):
        """(count(length == L), count(length == L and UNCERTAIN)) for L = 0..T (host sync)."""
        e = self.engine
        h = (C.c_int64 * (2 * (self.T + 1)))()
        L.check(e.lib.cmbpo_rollout_histogram(e.h, e._p(self.length), e._p(self.end_reason),
                                              self.B, self.T, h))
        a = np.frombuffer(h, dtype=np.int64).copy()
        return a[:self.T + 1], a[self.T + 1:]

    def truncate(self, cap_step=-1, cap_n=0, stop_step=-1):
        e = self.engine
        bufs = self.struct()
        L.check(e.lib.cmbpo_rollout_truncate(e.h, C.byref(bufs), self.B, self.T, int(cap_step),
                                             int(cap_n), int(stop_step)))

    def diagnostics(self):
        """cmbpo_rollout_diagnostics over the valid steps: dict of float64 sums / maxima (host sync);
        per-path returns / costs are left in self.path_return / self.path_cost (device, float64)."""
        e = self.engine
        st = (C.c_double * 8)()
        bufs = self.struct()
        L.check(e.lib.cmbpo_rollout_diagnostics(e.h, C.byref(bufs), self.B, e._p(self.path_return),
                                                e._p(self.path_cost), st))
        keys = ("rew", "cost", "val", "cval", "dyn_error", "max_dkl", "max_path_return", "n")
        return dict(zip(keys, (float(x) for x in st)))

    def gae(self, gamma, lam, cgamma, clam):
        """adv/ret/cadv/cret for every path from (length, last_val, last_cval)."""
        self.engine.gae_paths(self.rew, self.val, self.cost, self.cval, self.length, self.last_val,
                              self.last_cval, gamma, lam, cgamma, clam, self.B, self.T,
                              path_stride=1, time_stride=self.B,
                              out=(self.adv, self.ret, self.cadv, self.cret))

    # ---- reference-layout views (host) -------------------------------------------------
    def host(self, name):
        """Field `name` as the reference's [B, T, ...] numpy array."""
        x = getattr(self, name)
        if x.dim() == 3:
            return x.permute(1, 0, 2).contiguous().cpu().numpy()
        a = x.transpose(0, 1).contiguous().cpu().numpy()
        return a.astype(bool) if name == "term" else a

    def populated_mask(self):
        ln = self.length.cpu().numpy()
        return np.arange(self.T)[None, :] < ln[:, None]
