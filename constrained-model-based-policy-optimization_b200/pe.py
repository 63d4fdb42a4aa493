"""`B200PE`: the model contract FakeEnv and CPOPolicy consume (models/base_model.py:3-43,
models/pens/pe.py:401-434, 648-713), served by the CUDA ensemble-forward kernels.
"""
import itertools
import time
from collections import OrderedDict

import numpy as np

from . import _lib as L

_MOMENTS = ("mW", "vW", "mb", "vb")


def layer_decays(decay, n_layers):
    """Per-layer weight decay of build_PE (pe_factory.py:50-55): decay/4 on the first layer, decay on the last,
    decay/2 in between."""
    return [float(decay / 4 if l == 0 else (decay if l == n_layers - 1 else decay / 2)) for l in range(n_layers)]


class B200PE:
    """One ensemble living in an `Engine` slot (dynamics / V / VC).

    `predict_ensemble(x)` and `predict(x)` take and return numpy arrays like `PE` does
    (pe.py:648-713); the `*_device` variants keep everything on the GPU.
    """

    def __init__(self, engine, which, W, b, acts, probabilistic, elite_inds=(),
                 mu_in=None, var_in=None, mu_out=None, var_out=None, name="PE"):
        self.engine, self.which, self.name = engine, which, name
        self._probabilistic = bool(probabilistic)
        self.num_nets = int(W[0].shape[0])
        self._in_dim = int(W[0].shape[1])
        last = int(W[-1].shape[2])
        self._d = last // 2 if probabilistic else last
        self._model_inds = [int(i) for i in elite_inds]
        self.num_elites = len(self._model_inds)
        engine.set_network(which, W, b, acts, mu_in, var_in, mu_out, var_out,
                           probabilistic, self._model_inds)

    @classmethod
    def from_arrays(cls, engine, which, ens, name="PE"):
        """Build from a plain container with fields W, b, acts, probabilistic, mu_in, ..."""
        return cls(engine, which, ens.W, ens.b, ens.acts, ens.probabilistic, ens.elite_inds,
                   ens.mu_in, ens.var_in, ens.mu_out, ens.var_out, name=name)

    @classmethod
    def view(cls, engine, which, name="PE"):
        """A model object over a slot whose weights were already uploaded (Engine.set_network)."""
        meta = engine.nets[which]
        self = cls.__new__(cls)
        self.engine, self.which, self.name = engine, which, name
        self._probabilistic = meta["probabilistic"]
        self.num_nets, self._in_dim, self._d = meta["E"], meta["dims"][0], meta["D"]
        self._model_inds = list(meta["elite_inds"])
        self.num_elites = len(self._model_inds)
        return self

    # --- checkpoint and resume (checkpoint.save_state / load_state) ---
    def state_dict(self):
        """Everything a resumed run needs to continue this ensemble's training bit for bit, as numpy arrays and plain
        values: per layer W [E,in,out], b [E,out] and the Adam moments (absent before the first train()), the step
        count (-1: no optimiser state), the scalers as last uploaded, the elites and the training configuration
        with the running scaler statistics."""
        e = self.engine
        meta = e.nets[self.which]
        layers, step = [], -1
        for l in range(len(meta["dims"]) - 1):
            W, b = e.get_weights(self.which, l)
            mom, step = e.train_state_get(self.which, l)
            layer = {"W": W.cpu().numpy(), "b": b.cpu().numpy()}
            if mom is not None:
                layer.update(zip(_MOMENTS, (x.cpu().numpy() for x in mom)))
            layers.append(layer)
        train = None
        if hasattr(self, "_train_args"):
            train = dict(self._train_args)
            train["scaler_cache"] = {k: {"count": int(c), "mean": mu, "var": var}
                                     for k, (c, mu, var) in self._scaler_cache.items()}
        return {"name": self.name, "precision": e.precision_name, "dims": list(meta["dims"]),
                "acts": list(meta["acts"]), "probabilistic": self._probabilistic, "elite_inds": list(self._model_inds),
                "scalers": dict(meta["scalers"]), "layers": layers, "step": int(step), "train": train}

    @classmethod
    def from_state_dict(cls, engine, which, sd):
        """The inverse of state_dict() into slot `which` of `engine`: the weights first (a new set of weights drops the
        slot's optimiser state), then the optimiser state and the training configuration."""
        engine.check_precision(sd["precision"])
        dims, layers = [int(d) for d in sd["dims"]], sd["layers"]
        E = int(layers[0]["W"].shape[0]) if layers else 0
        if len(layers) != len(dims) - 1:
            raise ValueError("%d layers for dims %s" % (len(layers), dims))
        step = int(sd["step"])
        for l, layer in enumerate(layers):
            want = {"W": (E, dims[l], dims[l + 1]), "b": (E, dims[l + 1])}
            if step >= 0:
                want.update(mW=want["W"], vW=want["W"], mb=want["b"], vb=want["b"])
            for k, shape in want.items():
                if k not in layer or tuple(layer[k].shape) != shape:
                    raise ValueError("layer %d: %s is %s, dims %s want %s"
                                     % (l, k, None if k not in layer else tuple(layer[k].shape), dims, shape))
        sc = sd["scalers"]
        self = cls(engine, which, [x["W"] for x in layers], [x["b"] for x in layers], sd["acts"], sd["probabilistic"],
                   sd["elite_inds"], sc["mu_in"], sc["var_in"], sc["mu_out"], sc["var_out"], name=sd["name"])
        if sd["train"] is not None:
            args = dict(sd["train"])
            cache = args.pop("scaler_cache")
            self.configure_training(**args)
            self._scaler_cache = {k: (int(c["count"]), c["mean"], c["var"]) for k, c in cache.items()}
        if step >= 0:
            for l, x in enumerate(layers):
                engine.train_state_set(which, l, *(x[k] for k in _MOMENTS), step)
        return self

    # --- contract properties (pe.py:401-434) ---
    @property
    def elite_inds(self):
        return self._model_inds

    @property
    def is_probabilistic(self):
        return self._probabilistic

    @property
    def is_ensemble(self):
        return self.num_nets > 1

    @property
    def in_dim(self):
        return self._in_dim

    @property
    def out_dim(self):
        # pe.py:425-430: the reference returns None for a probabilistic ensemble (missing
        # `return`); FakeEnv.output_dim is never read, so mirror it.
        return None if self._probabilistic else self._d

    @property
    def is_tf_model(self):
        return False

    # --- prediction ---
    def predict_ensemble_device(self, x, precision=None):
        return self.engine.predict_ensemble(self.which, x, precision)

    def predict_device(self, x, precision=None):
        return self.engine.predict_mean(self.which, x, precision)

    def predict_ensemble(self, inputs, *args, **kwargs):
        """pe.py:671-713: 2-D inputs -> every member on the same rows; 3-D -> member i on slice i."""
        out = self.predict_ensemble_device(np.asarray(inputs, np.float32))
        if self._probabilistic:
            return out[0].cpu().numpy(), out[1].cpu().numpy()
        return out.cpu().numpy()

    def predict(self, inputs, *args, **kwargs):
        """pe.py:648-669."""
        inputs = np.asarray(inputs, np.float32)
        assert len(inputs.shape) == 2
        out = self.predict_device(inputs)
        if self._probabilistic:
            return [out[0].cpu().numpy(), out[1].cpu().numpy()]
        return out.cpu().numpy()

    # --- training (SURVEY.md 8f-4; models/pens/pe.py:457-646) ---
    def configure_training(self, loss=None, lr=1e-3, decay=1e-4, use_scaler_in=False, use_scaler_out=False,
                           math="fp32", n_layers=None):
        """What `build_PE` fixes at construction (pe_factory.py:9-60): loss type ('MSPE' for the probabilistic
        dynamics ensemble, 'MSE' for value ensembles), Adam learning rate, weight decay (first layer decay/4,
        hidden layers decay/2, last layer decay), which scalers `train` re-fits.  `math`: 'fp32' | 'tf32'
        (tensor-core GEMMs) | 'bf16' (tcgen05 GEMMs on bf16 operands, fp32 accumulation and optimiser state)."""
        if math not in L.TRAIN_MATHS:
            raise ValueError("math must be one of %s, not %r" % (", ".join(L.TRAIN_MATHS), math))
        if loss is None:
            loss = "MSPE" if self._probabilistic else "MSE"
        assert loss in ("MSPE", "MSE"), "losses of the CMBPO configs: MSPE (dynamics), MSE (V / VC)"
        nl = n_layers or (len(self.engine.nets[self.which]["dims"]) - 1)
        cfg = L.TrainCfg()
        cfg.loss = L.LOSS_MSPE if loss == "MSPE" else L.LOSS_MSE
        cfg.lr, cfg.beta1, cfg.beta2, cfg.eps = float(lr), 0.9, 0.999, 1e-8
        for l, wd in enumerate(layer_decays(decay, nl)):
            cfg.weight_decay[l] = wd
        cfg.math = L.TRAIN_MATHS[math]
        self._train_cfg = cfg
        self._train_args = dict(loss=loss, lr=float(lr), decay=float(decay), use_scaler_in=bool(use_scaler_in),
                                use_scaler_out=bool(use_scaler_out), math=math, n_layers=nl)
        self._use_scaler_in, self._use_scaler_out = bool(use_scaler_in), bool(use_scaler_out)
        self._scaler_cache = {"in": (0, None, None), "out": (0, None, None)}
        return self

    def _fit_scaler(self, key, data):
        """TensorStandardScaler.fit (pens/utils.py:119-138, 220-231): running merge of batch mean / variance."""
        count, mu, var = self._scaler_cache[key]
        b_mu = np.mean(data, axis=0, keepdims=True)
        b_var = np.var(data, axis=0, keepdims=True)
        n = data.shape[0]
        if mu is None:
            mu, var = np.zeros_like(b_mu), np.ones_like(b_var)
        delta = b_mu - mu
        tot = count + n
        new_mu = mu + delta * n / tot
        m2 = var * count + b_var * n + np.square(delta) * count * n / tot
        self._scaler_cache[key] = (tot, new_mu, m2 / tot)
        return new_mu.astype(np.float32), (m2 / tot).astype(np.float32)

    def _gather(self, src, idx, width):
        e = self.engine
        out = e.empty(idx.shape[0], idx.shape[1], width)
        L.check(e.lib.cmbpo_gather_rows(e.h, e._p(src), width, e._p(idx), idx.numel(), e._p(out)))
        return out

    def train(self, inputs, targets, batch_size=32, max_epochs=None, max_epochs_since_update=5,
              min_epoch_before_break=0, hide_progress=False, holdout_ratio=0.0, max_logging=5000,
              max_grad_updates=None, timer=None, max_t=None, rng=None, **kwargs):
        """PE.train (pe.py:457-646) on the device: holdout split, scaler fit, bootstrap indices per member
        (pe.py:523), epochs of Adam steps on [E, batch, .] slices, row shuffling between epochs, holdout loss and
        the early-stopping rule of `_save_best` (pe.py:367-389), elite selection by holdout loss (pe.py:396-399).
        Random draws come from `rng` (default: the global `np.random` stream, in the reference's call order).
        Returns OrderedDict({name/val_loss})."""
        assert hasattr(self, "_train_cfg"), "call configure_training() first"
        rng = rng or np.random
        e, t = self.engine, self.engine.torch
        E = self.num_nets
        inputs = np.asarray(inputs, np.float32)
        targets = np.asarray(targets, np.float32)
        self._max_epochs_since_update = max_epochs_since_update
        snapshots = {i: (None, 1e10) for i in range(E)}
        epochs_since_update = 0
        num_holdout = min(int(inputs.shape[0] * holdout_ratio), max_logging)
        permutation = rng.permutation(inputs.shape[0])
        inputs, hold_in = inputs[permutation[num_holdout:]], inputs[permutation[:num_holdout]]
        targets, hold_tg = targets[permutation[num_holdout:]], targets[permutation[:num_holdout]]
        if self._use_scaler_in or self._use_scaler_out:
            mi = vi = mo = vo = None
            if self._use_scaler_in:
                mi, vi = self._fit_scaler("in", inputs)
            if self._use_scaler_out:
                mo, vo = self._fit_scaler("out", targets)
            e.set_scalers(self.which, mi, vi, mo, vo)
        e.train_begin(self.which)
        d_in, d_tg = e.to_device(inputs, t.float32), e.to_device(targets, t.float32)
        n = inputs.shape[0]
        idxs = rng.randint(n, size=[E, n])
        if num_holdout:
            h_in = e.to_device(np.ascontiguousarray(np.broadcast_to(hold_in[None], (E,) + hold_in.shape)), t.float32)
            h_tg = e.to_device(np.ascontiguousarray(np.broadcast_to(hold_tg[None], (E,) + hold_tg.shape)), t.float32)
        epoch_iter = range(max_epochs) if max_epochs else itertools.count()
        t0 = time.time()
        grad_updates, break_train = 0, False
        Din, D = inputs.shape[1], targets.shape[1]
        for epoch in epoch_iter:
            d_idx = e.to_device(idxs.astype(np.int32), t.int32)
            for b0 in range(0, n, batch_size):
                bi = d_idx[:, b0:b0 + batch_size].contiguous()
                e.train_step(self.which, self._gather(d_in, bi, Din), self._gather(d_tg, bi, D), self._train_cfg)
                grad_updates += 1
            # shuffle_rows (pe.py:484-486)
            order = np.argsort(rng.uniform(size=idxs.shape), axis=-1)
            idxs = idxs[np.arange(E)[:, None], order]
            if not hide_progress and num_holdout:
                holdout_losses = e.train_loss(self.which, h_in, h_tg).cpu().numpy()
                updated = False
                for i in range(E):                                   # _save_best (pe.py:367-389)
                    best = snapshots[i][1]
                    if (best - holdout_losses[i]) / best > 0.01:
                        snapshots[i] = (epoch, float(holdout_losses[i]))
                        updated = True
                epochs_since_update = 0 if updated else epochs_since_update + 1
                break_train = epochs_since_update > max_epochs_since_update
            if (break_train and epoch > min_epoch_before_break) or (max_grad_updates and grad_updates > max_grad_updates):
                break
            if max_t and time.time() - t0 > max_t:
                break
        if num_holdout:
            holdout_losses = e.train_loss(self.which, h_in, h_tg).cpu().numpy()
        else:                      # np.sort of an empty feed would be nan in the reference; keep the old elites
            holdout_losses = np.zeros(E, np.float32)
        sorted_inds = np.argsort(holdout_losses)
        self._model_inds = sorted_inds[:self.num_elites].tolist() if num_holdout else self._model_inds
        e.train_end(self.which, self._model_inds)
        self._snapshots, self._grad_updates = snapshots, grad_updates
        val_loss = float(np.sort(holdout_losses)[:self.num_elites].mean())
        return OrderedDict({f"{self.name}/val_loss": val_loss})

    def validate(self, inputs, targets):
        """pe.py:440-451: mean holdout loss of the best `num_elites` members."""
        e, t = self.engine, self.engine.torch
        E = self.num_nets
        x = np.ascontiguousarray(np.broadcast_to(np.asarray(inputs, np.float32)[None], (E,) + tuple(np.shape(inputs))))
        y = np.ascontiguousarray(np.broadcast_to(np.asarray(targets, np.float32)[None], (E,) + tuple(np.shape(targets))))
        e.train_begin(self.which)
        losses = e.train_loss(self.which, e.to_device(x, t.float32), e.to_device(y, t.float32)).cpu().numpy()
        return float(np.sort(losses)[:self.num_elites].mean())
