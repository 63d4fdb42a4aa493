"""`B200Policy`: the inference side of CPOPolicy (policies/cpo_policy.py:801-835) on the GPU:
Gaussian actor (network/ac_network.py:99-123) + V and VC ensembles read through PE.predict.

Training (CPOAgent.update_pi, PE.train) is out of scope: after every policy / critic update
the trainer calls `load_actor` / `load_values` to refresh the device copies.
"""
import numpy as np

from . import _lib as L
from .pe import B200PE


class _Agent:
    reward_penalized = False      # cpo_policy.py:369; read by ModelSampler.finish_all_paths


class B200Policy:
    def __init__(self, engine, seed=0):
        self.engine = engine
        self.agent = _Agent()
        self.seed = int(seed)
        self._calls = 0
        self.v = self.vc = None
        self.log_std = None

    def load_actor(self, W, b, log_std):
        self.engine.set_actor(W, b, log_std)
        self.log_std = np.asarray(log_std, np.float32).copy()
        self.act_dim = int(self.log_std.shape[0])

    @property
    def log_std_device(self):
        """The actor's log_std variable [A] as a device tensor."""
        return self.engine.to_device(self.log_std, self.engine.torch.float32)

    def attach_loaded(self, log_std):
        """Use networks that were already uploaded to the engine (e.g. after an NCCL broadcast)."""
        self.log_std = np.asarray(log_std, np.float32).copy()
        self.act_dim = int(self.log_std.shape[0])
        self.v = B200PE.view(self.engine, L.NET_V, name="VEnsemble")
        self.vc = B200PE.view(self.engine, L.NET_VC, name="VCEnsemble")

    def load_values(self, v_ens, vc_ens):
        self.v = B200PE.from_arrays(self.engine, L.NET_V, v_ens, name="VEnsemble")
        self.vc = B200PE.from_arrays(self.engine, L.NET_VC, vc_ens, name="VCEnsemble")

    # ---- checkpoint and resume (checkpoint.save_state / load_state) ----------------------------
    def state_dict(self):
        """The actor (W [in,out], b [out] per layer, log_std), the seed and the call counter that key the actions'
        Philox draws.  V and VC are not part of it: save them with their own B200PE.state_dict()."""
        e = self.engine
        W, b = [], []
        for l in range(len(e.nets[L.NET_ACTOR]["dims"]) - 1):
            w, bb = e.get_weights(L.NET_ACTOR, l)
            W.append(w[0].cpu().numpy())
            b.append(bb[0].cpu().numpy())
        return {"precision": e.precision_name, "actor_W": W, "actor_b": b, "log_std": self.log_std.copy(),
                "seed": self.seed, "calls": self._calls}

    @classmethod
    def from_state_dict(cls, engine, sd, v=None, vc=None):
        """The inverse of state_dict().  Restore V and VC first (B200PE.from_state_dict into NET_V / NET_VC) and pass
        the objects that returns, or leave `v` / `vc` None to attach views of those slots, as attach_loaded does."""
        engine.check_precision(sd["precision"])
        if L.NET_V not in engine.nets or L.NET_VC not in engine.nets:
            raise L.CmbpoError("restore V and VC into the Engine before the policy")
        self = cls(engine, seed=sd["seed"])
        self.load_actor(sd["actor_W"], sd["actor_b"], sd["log_std"])
        self._calls = int(sd["calls"])
        self.v = v if v is not None else B200PE.view(engine, L.NET_V, name="VEnsemble")
        self.vc = vc if vc is not None else B200PE.view(engine, L.NET_VC, name="VCEnsemble")
        return self

    def reset(self):
        pass

    def get_action_outs(self, obs, eps=None):
        """cpo_policy.py:801-823.  `eps` injects the N(0,1) draws of ac_network.py:109;
        by default they come from the Philox stream keyed (seed, row, call counter)."""
        obs = np.asarray(obs, np.float32)
        single = obs.ndim == 1
        if single:
            obs = obs[None]
        out = self.engine.policy_act(obs, eps=eps, seed=self.seed, step=self._calls)
        self._calls += 1
        n = obs.shape[0]
        res = {"pi": out["pi"].cpu().numpy(), "logp_pi": out["logp"].cpu().numpy(),
               "pi_info": {"mu": out["mu"].cpu().numpy(),
                           "log_std": np.outer(np.ones(n, np.float32), self.log_std)},
               "v": out["v"].cpu().numpy(), "vc": out["vc"].cpu().numpy()}
        return res

    def get_v(self, obs):
        obs = np.asarray(obs, np.float32)
        if obs.ndim == 1:
            obs = obs[None]
        return self.engine.policy_act(obs, with_actor=False)["v"].cpu().numpy()

    def get_vc(self, obs):
        obs = np.asarray(obs, np.float32)
        if obs.ndim == 1:
            obs = obs[None]
        return self.engine.policy_act(obs, with_actor=False)["vc"].cpu().numpy()
