"""`CPOBuffer` store / finish_path / get (buffers/cpobuffer.py:160-290) for the flat on-policy
layout.  Real-environment samples arrive one step at a time from MuJoCo on the host, so rows are
staged in host arrays exactly like the reference; the GAE / cost-GAE scans of `finish_path` and
the advantage normalisation of `get()` run on the GPU (cmbpo_gae_flat, cmbpo_adv_*).

The off-policy archive and its sampling helpers (cpobuffer.py:210-248, 292-534) are host
bookkeeping outside the accelerated path and are not reproduced (SURVEY.md section 8a, row a9).
"""
import numpy as np

from . import _lib as L

EPS = 1e-8


class CPOBuffer:
    def __init__(self, size, archive_size, observation_space, action_space, engine=None,
                 *args, **kwargs):
        if engine is None:
            raise L.CmbpoError("CPOBuffer needs the Engine that runs its scans")
        self.engine = engine
        self.obs_shape = tuple(observation_space.shape)
        self.act_shape = tuple(action_space.shape)
        self.archive_size = archive_size
        self.max_size = int(size)
        self.gamma, self.lam, self.cost_gamma, self.cost_lam = 0.99, 0.95, 0.99, 0.95
        self.scan_mode = L.SCAN_STRICT
        self.pi_info_bufs = {}
        self.sorted_pi_info_keys = []
        self.reset_buffers()

    def initialize(self, pi_info_shapes, gamma=0.99, lam=0.95, cost_gamma=0.99, cost_lam=0.95):
        self.pi_info_shapes = dict(pi_info_shapes)
        self.pi_info_bufs = {k: np.zeros([self.max_size] + list(v), dtype=np.float32)
                             for k, v in pi_info_shapes.items()}
        self.sorted_pi_info_keys = sorted(self.pi_info_bufs)
        self.gamma, self.lam = gamma, lam
        self.cost_gamma, self.cost_lam = cost_gamma, cost_lam

    def reset_buffers(self):
        n = self.max_size
        f = lambda *s: np.zeros((n,) + s, dtype=np.float32)
        self.obs_buf, self.nextobs_buf, self.act_buf = f(*self.obs_shape), f(*self.obs_shape), f(*self.act_shape)
        self.adv_buf, self.rew_buf, self.val_buf, self.ret_buf = f(), f(), f(), f()
        self.cadv_buf, self.cost_buf, self.cret_buf, self.cval_buf = f(), f(), f(), f()
        self.logp_buf = f()
        self.term_buf = np.zeros(n, dtype=bool)
        self.epoch_buf = np.ones(n, dtype=np.float32) * -1
        for k in self.pi_info_bufs:
            self.pi_info_bufs[k] = np.zeros_like(self.pi_info_bufs[k])
        self.ptr, self.path_start_idx, self.path_finished = 0, 0, False
        self._pending = []          # (start, stop, last_val, last_cval) of paths not yet scanned

    @property
    def size(self):
        return self.ptr

    def store(self, obs, act, next_obs, rew, val, cost, cval, logp, pi_info, term, epoch):
        """cpobuffer.py:160-176."""
        assert self.ptr < self.max_size
        p = self.ptr
        self.obs_buf[p], self.act_buf[p], self.nextobs_buf[p] = obs, act, next_obs
        self.rew_buf[p], self.val_buf[p], self.cost_buf[p], self.cval_buf[p] = rew, val, cost, cval
        self.logp_buf[p], self.term_buf[p], self.epoch_buf[p] = logp, term, epoch
        for k in self.sorted_pi_info_keys:
            self.pi_info_bufs[k][p] = pi_info[k]
        self.ptr += 1
        self.path_finished = False

    def finish_path(self, last_val=0, last_cval=0, defer=False):
        """cpobuffer.py:179-207.  `defer=True` queues the path so that several paths are scanned
        by one launch (flush_paths); results are identical."""
        self._pending.append((self.path_start_idx, self.ptr, float(np.squeeze(last_val)),
                              float(np.squeeze(last_cval))))
        self.path_start_idx = self.ptr
        self.path_finished = True
        if not defer:
            self.flush_paths()

    def flush_paths(self):
        if not self._pending:
            return
        e, t = self.engine, self.engine.torch
        lo, hi = self._pending[0][0], self._pending[-1][1]
        offs = np.array([p[0] - lo for p in self._pending] + [hi - lo], dtype=np.int64)
        lv = np.array([p[2] for p in self._pending], dtype=np.float32)
        lc = np.array([p[3] for p in self._pending], dtype=np.float32)
        self._pending = []
        if hi == lo:
            return
        s = slice(lo, hi)
        dev = lambda a: e.to_device(a[s], t.float32)
        adv, ret, cadv, cret = e.gae_flat(dev(self.rew_buf), dev(self.val_buf), dev(self.cost_buf),
                                          dev(self.cval_buf), e.to_device(offs, t.int64),
                                          e.to_device(lv), e.to_device(lc), self.gamma, self.lam,
                                          self.cost_gamma, self.cost_lam, scan=self.scan_mode)
        self.adv_buf[s], self.ret_buf[s] = adv.cpu().numpy(), ret.cpu().numpy()
        self.cadv_buf[s], self.cret_buf[s] = cadv.cpu().numpy(), cret.cpu().numpy()

    def get(self):
        """cpobuffer.py:249-290 (without the archive dump)."""
        self.flush_paths()
        e, t = self.engine, self.engine.torch
        n = self.ptr
        if n > 0:
            adv, cadv = e.to_device(self.adv_buf[:n]), e.to_device(self.cadv_buf[:n])
            ret, cret = e.to_device(self.ret_buf[:n]), e.to_device(self.cret_buf[:n])
            sums = e.adv_statistics_device(adv, cadv, ret, cret, 1, n, n, 1, None)
            e.adv_normalise_device(adv, cadv, 1, n, n, 1, None, sums)
            st = e.stats_from_sums(sums.cpu().numpy())
            self.adv_buf[:n], self.cadv_buf[:n] = adv.cpu().numpy(), cadv.cpu().numpy()
            ret_mean, cret_mean = st["ret_mean"], st["cret_mean"]
        else:
            ret_mean = cret_mean = 0
        res = [self.obs_buf, self.act_buf, self.adv_buf, self.cadv_buf, self.ret_buf, self.cret_buf,
               self.logp_buf, self.val_buf, self.cval_buf, self.cost_buf] + \
              [self.pi_info_bufs[k] for k in self.sorted_pi_info_keys]
        res = [v.copy()[:n] for v in res]
        diagnostics = dict(poolr_ret_mean=ret_mean, poolr_cret_mean=cret_mean)
        self.reset_buffers()
        return res, diagnostics
