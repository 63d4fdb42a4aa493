"""`Engine`: one library context on one B200, holding the four networks of a CMBPO rollout
(dynamics PE, actor, V ensemble, VC ensemble) and exposing the C ABI with torch device
tensors as arguments.  torch is used for device memory, streams and NCCL only.
"""
import ctypes as C

import numpy as np

from . import _lib as L
from .dist import combine_pass1, combine_pass2


def _as_f32(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float32))


def _host_row(a):
    """A [1, n] float32 host copy of a scaler vector (numpy array or tensor), None for None."""
    if a is None:
        return None
    if hasattr(a, "is_cuda"):
        a = a.detach().cpu().numpy()
    return _as_f32(a).reshape(1, -1).copy()


class Engine:
    def __init__(self, device=0, precision="fp32"):
        import torch
        if not torch.cuda.is_available():
            raise L.CmbpoError("no CUDA device visible: cmbpo_b200 has no CPU fallback")
        self.torch = torch
        self.lib = L.load()
        self.device_index = int(device)
        self.device = torch.device("cuda", self.device_index)
        self.precision = L.PRECISIONS[precision] if isinstance(precision, str) else int(precision)
        h = C.c_void_p()
        L.check(self.lib.cmbpo_ctx_create(self.device_index, C.byref(h)))
        self.h = h
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
        L.check(self.lib.cmbpo_ctx_set_stream(self.h, C.c_void_p(stream)))
        self.nets = {}

    def close(self):
        if getattr(self, "h", None):
            self.lib.cmbpo_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ helpers
    def _p(self, t, dtype=None):
        """device pointer of a contiguous tensor on this engine's device (None -> NULL)."""
        if t is None:
            return None
        assert t.is_cuda and t.device.index == self.device_index, "tensor on the wrong device"
        assert t.is_contiguous(), "tensor must be contiguous"
        if dtype is not None:
            assert t.dtype == dtype, "expected %s got %s" % (dtype, t.dtype)
        return C.c_void_p(t.data_ptr())

    def to_device(self, a, dtype=None):
        t = self.torch
        if isinstance(a, t.Tensor):
            x = a.to(self.device)
            if dtype is not None:
                x = x.to(dtype)
            return x.contiguous()
        arr = np.ascontiguousarray(a)
        if arr.nbytes >= (1 << 20) and arr.dtype == np.float32 and (dtype is None or dtype == t.float32):
            # large pageable arrays (the start states of a rollout): one host copy into a cached page-locked block and
            # one DMA, instead of the driver's chunked bounce-buffer path for pageable memory (~3x slower)
            stage = getattr(self, "_h2d_stage", None)
            if stage is None or stage.numel() < arr.size:
                stage = self._h2d_stage = t.empty(arr.size, dtype=t.float32, pin_memory=True)
                self._h2d_done = None
            if self._h2d_done is not None:
                self._h2d_done.synchronize()           # the previous upload out of this block has finished
            view = stage[:arr.size].view(arr.shape)
            view.copy_(t.from_numpy(arr))
            x = view.to(self.device, non_blocking=True)
            self._h2d_done = t.cuda.Event()
            self._h2d_done.record()
            return x
        x = t.from_numpy(arr).to(self.device, non_blocking=False)
        if dtype is not None:
            x = x.to(dtype)
        return x

    def empty(self, *shape, dtype=None):
        t = self.torch
        return t.empty(shape, dtype=dtype or t.float32, device=self.device)

    def zeros(self, *shape, dtype=None):
        t = self.torch
        return t.zeros(shape, dtype=dtype or t.float32, device=self.device)

    def synchronize(self):
        L.check(self.lib.cmbpo_ctx_synchronize(self.h))

    @property
    def precision_name(self):
        return {v: k for k, v in L.PRECISIONS.items()}[self.precision]

    def check_precision(self, recorded):
        """Refuse state saved from an Engine of another rollout precision: resumed on this one, the run would not
        continue the rollouts it was doing."""
        if recorded != self.precision_name:
            raise ValueError("the state was saved at rollout precision %r, this Engine runs %r"
                             % (recorded, self.precision_name))

    @property
    def launch_count(self):
        return int(self.lib.cmbpo_ctx_launch_count(self.h))

    def profile(self, enable=True):
        """Bracket the dominant kernels (dynamics GEMM chain, GAE scan) with CUDA events."""
        L.check(self.lib.cmbpo_ctx_profile(self.h, int(enable)))

    def profile_read(self, slot, reset=True):
        """(summed device ms, launches) of slot 0 = dynamics GEMM chain, 1 = GAE scan."""
        ms, n = C.c_double(), C.c_int64()
        L.check(self.lib.cmbpo_ctx_profile_read(self.h, slot, C.byref(ms), C.byref(n), int(reset)))
        return ms.value, n.value

    # ------------------------------------------------------------------ weights
    def set_network(self, which, W, b, acts, mu_in=None, var_in=None, mu_out=None, var_out=None,
                    probabilistic=False, elite_inds=()):
        """W[l]: [E,in,out]; b[l]: [E,1,out] or [E,out]; numpy arrays or device tensors."""
        t = self.torch
        on_device = isinstance(W[0], t.Tensor)
        n_layers = len(W)
        E = int(W[0].shape[0])
        dims = [int(W[0].shape[1])] + [int(w.shape[2]) for w in W]
        keep = []   # keep host/device arrays alive across the call

        def ptr(a):
            if a is None:
                return None
            if on_device:
                x = a.to(self.device, t.float32).contiguous()
                keep.append(x)
                return x.data_ptr()
            x = _as_f32(a)
            keep.append(x)
            return x.ctypes.data

        Wp = (C.c_void_p * n_layers)(*[ptr(w) for w in W])
        bp = (C.c_void_p * n_layers)(*[ptr(x.reshape(E, -1)) for x in b])
        actsp = (C.c_int * n_layers)(*[L.ACT_IDS[a] for a in acts])
        dimsp = (C.c_int * (n_layers + 1))(*dims)
        elite = [int(i) for i in elite_inds]
        elp = (C.c_int * max(1, len(elite)))(*elite) if elite else (C.c_int * 1)(0)
        sc = [ptr(None if a is None else (a.reshape(-1)))
              for a in (mu_in, var_in, mu_out, var_out)]
        L.check(self.lib.cmbpo_net_set_weights(
            self.h, which, E, n_layers, dimsp, Wp, bp, actsp,
            C.c_void_p(sc[0]), C.c_void_p(sc[1]), C.c_void_p(sc[2]), C.c_void_p(sc[3]),
            int(bool(probabilistic)), elp, len(elite), int(on_device)))
        last = dims[-1]
        # the scalers as uploaded (the library keeps sigma = max(sqrt(var), 1e-2), not the variance): checkpoints
        # write these
        scalers = {k: _host_row(a) for k, a in zip(("mu_in", "var_in", "mu_out", "var_out"),
                                                   (mu_in, var_in, mu_out, var_out))}
        self.nets[which] = dict(E=E, dims=dims, D=last // 2 if probabilistic else last,
                                probabilistic=bool(probabilistic), elite_inds=elite, acts=list(acts),
                                scalers=scalers)

    # ------------------------------------------------------------------ ensemble training (SURVEY.md 8f-4)
    def train_begin(self, which):
        L.check(self.lib.cmbpo_ens_train_begin(self.h, which))

    def train_step(self, which, x, y, cfg, loss_out=None):
        """One Adam step of slot `which` on x [E,bs,in], y [E,bs,D] (device tensors, member e on slice e)."""
        t = self.torch
        x = self.to_device(x, t.float32)
        y = self.to_device(y, t.float32)
        assert x.dim() == 3 and y.dim() == 3 and x.shape[:2] == y.shape[:2]
        L.check(self.lib.cmbpo_ens_train_step(self.h, which, self._p(x), self._p(y), int(x.shape[1]), C.byref(cfg),
                                              self._p(loss_out)))

    def train_loss(self, which, x, y):
        """`self.loss` of the reference (pe.py:264): [E] device tensor of mean 0.5 (mean - transform(y))^2."""
        t = self.torch
        x = self.to_device(x, t.float32)
        y = self.to_device(y, t.float32)
        out = self.empty(int(x.shape[0]))
        L.check(self.lib.cmbpo_ens_train_loss(self.h, which, self._p(x), self._p(y), int(x.shape[1]), self._p(out)))
        return out

    def train_grads(self, which, layer):
        m = self.nets[which]
        dW = self.empty(m["E"], m["dims"][layer], m["dims"][layer + 1])
        db = self.empty(m["E"], m["dims"][layer + 1])
        L.check(self.lib.cmbpo_ens_train_grads(self.h, which, layer, self._p(dW), self._p(db)))
        return dW, db

    def get_weights(self, which, layer):
        m = self.nets[which]
        W = self.empty(m["E"], m["dims"][layer], m["dims"][layer + 1])
        b = self.empty(m["E"], m["dims"][layer + 1])
        L.check(self.lib.cmbpo_net_get_weights(self.h, which, layer, self._p(W), self._p(b)))
        return W, b

    def set_scalers(self, which, mu_in=None, var_in=None, mu_out=None, var_out=None):
        keep = [None if a is None else _as_f32(np.asarray(a).reshape(-1)) for a in (mu_in, var_in, mu_out, var_out)]
        p = [C.c_void_p(None if a is None else a.ctypes.data) for a in keep]
        L.check(self.lib.cmbpo_net_set_scalers(self.h, which, *p))
        sc = self.nets[which]["scalers"]
        for k, a in zip(("mu_in", "var_in", "mu_out", "var_out"), (mu_in, var_in, mu_out, var_out)):
            if a is not None:
                sc[k] = _host_row(a)

    def train_state_get(self, which, layer):
        """Checkpointing: ((mW, vW, mb, vb) device tensors, step count) of one layer of slot `which`'s optimiser
        state, or (None, -1) when the slot has none."""
        m = self.nets[which]
        E, K, H = m["E"], m["dims"][layer], m["dims"][layer + 1]
        mom = (self.empty(E, K, H), self.empty(E, K, H), self.empty(E, H), self.empty(E, H))
        step = C.c_int64()
        L.check(self.lib.cmbpo_ens_train_state_get(self.h, which, layer, *(self._p(x) for x in mom), C.byref(step)))
        return (mom if step.value >= 0 else None), step.value

    def train_state_set(self, which, layer, mW, vW, mb, vb, step):
        """Restore one layer's Adam moments and the slot's step count (creating the optimiser state if absent).
        Call after set_network, which drops the optimiser state."""
        t = self.torch
        m = self.nets[which]
        E, K, H = m["E"], m["dims"][layer], m["dims"][layer + 1]
        mom = [self.to_device(x, t.float32) for x in (mW, vW, mb, vb)]
        for x, shape in zip(mom, ((E, K, H), (E, K, H), (E, H), (E, H))):
            if tuple(x.shape) != shape:
                raise ValueError("Adam moment of shape %s for layer %d of shape %s" % (tuple(x.shape), layer, shape))
        L.check(self.lib.cmbpo_ens_train_state_set(self.h, which, layer, *(self._p(x) for x in mom), int(step)))

    def train_end(self, which, elite_inds=None):
        el = None if elite_inds is None else [int(i) for i in elite_inds]
        arr = (C.c_int * max(1, len(el or [])))(*(el or [0]))
        L.check(self.lib.cmbpo_ens_train_end(self.h, which, arr if el else None, len(el or [])))
        if el:
            self.nets[which]["elite_inds"] = el

    def set_actor(self, W, b, log_std):
        """W[l]: [in,out] dense kernels, tanh hidden, linear output (ac_network.py:26-33)."""
        t = self.torch
        if isinstance(W[0], t.Tensor):
            W3 = [w.unsqueeze(0) for w in W]
            b3 = [x.reshape(1, -1) for x in b]
            ls = log_std.to(self.device, t.float32).contiguous()
            lsp, dev = ls.data_ptr(), 1
        else:
            W3 = [np.asarray(w, np.float32)[None] for w in W]
            b3 = [np.asarray(x, np.float32).reshape(1, -1) for x in b]
            ls = _as_f32(log_std)
            lsp, dev = ls.ctypes.data, 0
        acts = ["tanh"] * (len(W) - 1) + [None]
        self.set_network(L.NET_ACTOR, W3, b3, acts)
        L.check(self.lib.cmbpo_actor_set_log_std(self.h, C.c_void_p(lsp), int(ls.shape[0]), dev))
        self.act_dim = int(ls.shape[0])

    # ------------------------------------------------------------------ forward passes
    def predict_ensemble(self, which, x, precision=None):
        t = self.torch
        net = self.nets[which]
        x = self.to_device(x, t.float32)
        is3d = x.dim() == 3
        N = x.shape[-2]
        mean = self.empty(net["E"], N, net["D"])
        var = self.empty(net["E"], N, net["D"]) if net["probabilistic"] else None
        L.check(self.lib.cmbpo_ens_predict(self.h, which, self._p(x), N, int(is3d), self._p(mean),
                                           self._p(var), self._prec(precision)))
        return (mean, var) if var is not None else mean

    def predict_mean(self, which, x, precision=None):
        t = self.torch
        net = self.nets[which]
        x = self.to_device(x, t.float32)
        N = x.shape[0]
        mean = self.empty(N, net["D"])
        var = self.empty(N, net["D"]) if net["probabilistic"] else None
        L.check(self.lib.cmbpo_ens_predict_mean(self.h, which, self._p(x), N, self._p(mean),
                                                self._p(var), self._prec(precision)))
        return (mean, var) if var is not None else mean

    def _prec(self, precision):
        if precision is None:
            return self.precision
        return L.PRECISIONS[precision] if isinstance(precision, str) else int(precision)

    def policy_act(self, obs, eps=None, path_ids=None, seed=0, step=0, precision=None,
                   with_actor=True):
        t = self.torch
        obs = self.to_device(obs, t.float32)
        N = obs.shape[0]
        A = self.act_dim if with_actor else 0
        pi = self.empty(N, A) if with_actor else None
        mu = self.empty(N, A) if with_actor else None
        logp = self.empty(N) if with_actor else None
        v, vc = self.empty(N), self.empty(N)
        eps = None if eps is None else self.to_device(eps, t.float32)
        path_ids = None if path_ids is None else self.to_device(path_ids, t.int32)
        L.check(self.lib.cmbpo_policy_act(self.h, self._p(obs), N, self._p(eps), self._p(path_ids),
                                          int(seed), int(step), self._p(pi), self._p(logp),
                                          self._p(mu), self._p(v), self._p(vc),
                                          self._prec(precision)))
        return dict(pi=pi, logp=logp, mu=mu, v=v, vc=vc)

    def fakeenv_step(self, cfg: L.EnvCfg, obs, act, elite_pos=None, state_eps=None, path_ids=None,
                     seed=0, step=0, precision=None):
        t = self.torch
        obs = self.to_device(obs, t.float32)
        act = self.to_device(act, t.float32)
        N, O = obs.shape
        elite_pos = None if elite_pos is None else self.to_device(elite_pos, t.int32)
        state_eps = None if state_eps is None else self.to_device(state_eps, t.float32)
        path_ids = None if path_ids is None else self.to_device(path_ids, t.int32)
        out = dict(next_obs=self.empty(N, O), rew=self.empty(N), cost=self.empty(N),
                   term=self.empty(N, dtype=t.uint8), dkl_path=self.empty(N),
                   ep_var=self.empty(N, O), dkl_mean=self.empty(1))
        L.check(self.lib.cmbpo_fakeenv_step(
            self.h, C.byref(cfg), self._p(obs), self._p(act), N, self._p(elite_pos),
            self._p(state_eps), self._p(path_ids), int(seed), int(step), self._p(out["next_obs"]),
            self._p(out["rew"]), self._p(out["cost"]), self._p(out["term"]),
            self._p(out["dkl_path"]), self._p(out["ep_var"]), self._p(out["dkl_mean"]),
            self._prec(precision)))
        return out

    # ------------------------------------------------------------------ GAE
    def gae_paths(self, rew, val, cost, cval, length, last_val, last_cval, gamma, lam, cgamma, clam,
                  n_paths, max_len, path_stride, time_stride, out=None):
        t = self.torch
        if out is None:
            out = tuple(t.zeros_like(rew) for _ in range(4))
        adv, ret, cadv, cret = out
        L.check(self.lib.cmbpo_gae_paths(
            self.h, self._p(rew), self._p(val), self._p(cost), self._p(cval), n_paths, max_len,
            path_stride, time_stride, self._p(length), self._p(last_val), self._p(last_cval),
            float(gamma), float(lam), float(cgamma), float(clam), self._p(adv), self._p(ret),
            self._p(cadv), self._p(cret)))
        return adv, ret, cadv, cret

    def gae_flat(self, rew, val, cost, cval, seg_offsets, last_val, last_cval, gamma, lam, cgamma,
                 clam, out=None, scan=L.SCAN_WARP):
        t = self.torch
        if out is None:
            out = tuple(t.zeros_like(rew) for _ in range(4))
        adv, ret, cadv, cret = out
        n_seg = seg_offsets.shape[0] - 1
        L.check(self.lib.cmbpo_gae_flat(
            self.h, self._p(rew), self._p(val), self._p(cost), self._p(cval),
            self._p(seg_offsets, t.int64), n_seg, self._p(last_val), self._p(last_cval),
            float(gamma), float(lam), float(cgamma), float(clam), self._p(adv), self._p(ret),
            self._p(cadv), self._p(cret), int(scan)))
        return adv, ret, cadv, cret

    def adv_statistics_device(self, adv, cadv, ret, cret, n_paths, max_len, path_stride, time_stride,
                              length, reduce_fn=None):
        """Two-pass float32 statistics of mpi_statistics_scalar (mpi_tools.py:71-92) with the sums kept on the
        device: no host synchronisation, so the host can queue the normalisation and whatever follows without
        waiting for the scans; with N > 1 the ranks meet only in the two all-reduces.  `reduce_fn(tensor)`
        all-reduces a small float64 tensor in place (multi-GPU).  Returns the device tensor of 8 float64 sums
        (see `stats_from_sums`)."""
        t = self.torch
        sums = self.zeros(8, dtype=t.float64)
        L.check(self.lib.cmbpo_adv_stats_pass1(self.h, self._p(adv), self._p(cadv), self._p(ret),
                                               self._p(cret), n_paths, max_len, path_stride,
                                               time_stride, self._p(length), self._p(sums)))
        if reduce_fn is not None:
            reduce_fn(sums)
        L.check(self.lib.cmbpo_adv_stats_pass2(self.h, self._p(adv), n_paths, max_len, path_stride,
                                               time_stride, self._p(length), self._p(sums), self._p(sums)))
        if reduce_fn is not None:
            reduce_fn(sums[5:6])                 # in place: a one-element view of the same memory
        return sums

    def adv_normalise_device(self, adv, cadv, n_paths, max_len, path_stride, time_stride, length, sums):
        """adv <- (adv - mean) / (std + 1e-8), cadv <- cadv - cmean from the device sums of
        `adv_statistics_device` (modelbuffer.py:196-204)."""
        L.check(self.lib.cmbpo_adv_normalise(self.h, self._p(adv), self._p(cadv), n_paths, max_len,
                                             path_stride, time_stride, self._p(length), self._p(sums)))

    @staticmethod
    def stats_from_sums(s):
        """dict of n, adv_mean, adv_std, cadv_mean, ret_mean, cret_mean (float32) from a HOST copy of the 8
        sums of adv_statistics_device()."""
        st = combine_pass1(s)
        st["adv_std"] = np.float32(combine_pass2(float(s[5]), st["n"])) if st["n"] else np.float32(0)
        return st

    def path_offsets(self, length):
        t = self.torch
        B = length.shape[0]
        off = self.empty(B + 1, dtype=t.int64)
        L.check(self.lib.cmbpo_path_offsets(self.h, self._p(length, t.int32), B, self._p(off)))
        return off

    def compact(self, field, B, T, width, length, offsets, n_rows, out=None):
        if out is None:
            out = self.empty(n_rows, width) if width > 1 or field.dim() == 3 else self.empty(n_rows)
        L.check(self.lib.cmbpo_compact_field(self.h, self._p(field), B, T, width, self._p(length),
                                             self._p(offsets), self._p(out)))
        return out

    def scatter_rows(self, dst, B, width, t_col, path_idx, src):
        n = path_idx.shape[0]
        L.check(self.lib.cmbpo_scatter_rows(self.h, self._p(dst), B, width, int(t_col),
                                            self._p(path_idx), self._p(src), n))
