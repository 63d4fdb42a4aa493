"""-m gpu: the bf16 ensemble training step (cmbpo_train_cfg.math = CMBPO_TRAIN_BF16, csrc/train_tc.cu) against two
oracles: the bf16-rounding restatement (tests/train_oracle_bf16.py, rounding where the kernels round) and the plain
float64 step (oracle/train_oracle.py).  Three Adam steps per shape: the loss vector at every step, dW / db of every
layer at step 0 (the last layer's dW isolates the forward and weight-gradient GEMMs; earlier layers add the
data-gradient GEMM).  Also: bit-identical repeats, W16 rebuilt after fp32 / TF32 steps, the launch count, the
B200PE.train loop, and the rejection of unknown `math` values.

Residuals are max |got - want| / max |want| over the tensor (per-member relative error for the loss vector).
Bounds are about twice the largest residual measured over these cases on a B200; the measured values are:
  against the rounding oracle:  loss 2.1e-7 .. 1.8e-5, dW 0 .. 1.4e-3, db 4.0e-7 .. 4.4e-4;
  against float64:              loss 9.9e-6 .. 3.8e-4, dW 3.5e-3 .. 6.0e-3, db 3.2e-3 .. 9.4e-3
(NVIDIA B200, 1000 W power limit).  Weights and biases after the three steps: 0.84 .. 1.0 of each layer's
elements are within 1e-6 of the rounding oracle's; against oracles without the decay or with a 10 % larger
learning rate at most 0.12 are, so the bound 0.6 tells a correct fused Adam update from a wrong one.
The interleaving test checks its bf16 steps against the float64-oracle bounds:
a stale W16 there misses an Adam step of lr = 1e-2, tens of percent of a weight.
"""
import numpy as np
import pytest

from oracle import cmbpo_oracle as orc
from oracle import train_oracle as tro
import train_oracle_bf16 as trb

pytestmark = pytest.mark.gpu

# (rounding oracle, float64 oracle) bounds per quantity
BOUND = {"loss": (4e-5, 8e-4), "dW": (3e-3, 1.2e-2), "db": (1e-3, 2e-2)}
# weights and biases after three Adam steps: at least ADAM_FRAC of each layer's elements within ADAM_ATOL
ADAM_ATOL, ADAM_FRAC = 1e-6, 0.6
# fp32 / TF32 bounds of tests/test_gpu_train.py, for the steps of the interleaving test that are not bf16
OTHER = {"fp32": (2e-5, 2e-4), "tf32": (2e-3, 5e-3)}

# name: E, O, A, hidden, probabilistic, bs, activation
CASES = {
    "hcs": (7, 17, 6, (512, 512), True, 256, "swish"),
    "humanoid": (7, 47, 17, (200, 200, 200, 200), True, 256, "swish"),
    "hc_o20_bs100": (7, 20, 6, (512, 512), True, 100, "swish"),
    "v_mse": (3, 17, 6, (128, 128), False, 256, "swish"),
    "e1_bs1_tanh": (1, 17, 6, (256, 256), True, 1, "tanh"),
    "e8_bs257_tanh": (8, 17, 6, (200, 200), True, 257, "tanh"),
    "e1_bs1000": (1, 17, 6, (512, 512), True, 1000, "swish"),
    "v_bs1000_tanh": (3, 17, 6, (128, 128), False, 1000, "tanh"),
}


def _setup(engine, seed, E, bs, O, A, hidden, prob=True, act="swish"):
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    rng = np.random.default_rng(seed)
    Din, D = O + A, O + 1
    if prob:
        dyn, _, _, _ = orc.make_problem(seed, O, A, hidden=hidden, num_nets=E, num_elites=max(1, E - 2))
        ens, which = dyn, L.NET_DYN
    else:
        _, _, v, _ = orc.make_problem(seed, O, A, hidden=(64, 64), vf_nets=E, vf_hidden=hidden)
        ens, which, Din, D = v, L.NET_V, O, 1
    ens.acts[:] = [act] * (len(ens.acts) - 1) + [None]
    for bl in ens.b:                                   # non-zero biases so that their gradients matter
        bl += 0.05 * rng.standard_normal(bl.shape).astype(np.float32)
    model = cb.B200PE.from_arrays(engine, which, ens)  # a new set of weights: a fresh optimiser state
    x = (rng.standard_normal((E, bs, Din)) * np.maximum(np.sqrt(ens.var_in), 1e-2) + ens.mu_in).astype(np.float32)
    y = (rng.standard_normal((E, bs, D)) * np.maximum(np.sqrt(ens.var_out), 1e-2) + ens.mu_out).astype(np.float32)
    return model, ens, which, x, y


def _f64(ens):
    return ([w.astype(np.float64) for w in ens.W], [b.astype(np.float64).reshape(b.shape[0], -1) for b in ens.b],
            dict(mu_in=ens.mu_in.astype(np.float64), var_in=ens.var_in.astype(np.float64),
                 mu_out=ens.mu_out.astype(np.float64), var_out=ens.var_out.astype(np.float64)))


def _rel(got, want):
    return float(np.abs(got - want).max() / np.abs(want).max())


def _loss_rel(got, want):
    return float((np.abs(got - want) / np.abs(want)).max())


def _case(engine, name, seed=11):
    E, O, A, hidden, prob, bs, act = CASES[name]
    model, ens, which, x, y = _setup(engine, seed, E, bs, O, A, hidden, prob, act)
    return model, ens, which, x, y, ("MSPE" if prob else "MSE")


@pytest.mark.parametrize("name", list(CASES))
def test_bf16_steps_vs_oracles(engine, name):
    model, ens, which, x, y, loss = _case(engine, name)
    decay = 1e-2
    model.configure_training(loss=loss, lr=1e-3, decay=decay, math="bf16")
    engine.train_begin(which)
    W, b, sc = _f64(ens)
    nl = len(W)
    opts = [tro.Adam([p for l in range(nl) for p in (W[l], b[l])], lr=1e-3) for _ in range(2)]
    state = [(W, b), (W, b)]                           # rounding oracle, float64 oracle: each its own trajectory
    x64, y64 = x.astype(np.float64), y.astype(np.float64)
    lout = engine.empty(ens.W[0].shape[0])
    worst = {k: [0.0, 0.0] for k in BOUND}
    for step in range(3):
        ref = [trb.train_step(*state[0], ens.acts, x64, y64, loss, opts[0], decay, round_bf16=True, **sc),
               tro.train_step(*state[1], ens.acts, x64, y64, loss, opts[1], decay, **sc)]
        engine.train_step(which, x, y, model._train_cfg, lout)
        got_l = lout.cpu().numpy()
        for k in range(2):
            worst["loss"][k] = max(worst["loss"][k], _loss_rel(got_l, ref[k][0]))
        if step == 0:
            for l in range(nl):
                dW, db = engine.train_grads(which, l)
                dW, db = dW.cpu().numpy(), db.cpu().numpy()
                for k in range(2):
                    worst["dW"][k] = max(worst["dW"][k], _rel(dW, ref[k][3][l]))
                    worst["db"][k] = max(worst["db"][k], _rel(db, ref[k][4][l]))
        state = [(r[1], r[2]) for r in ref]
    print("bf16 residuals %s: %s" % (name, " ".join("%s %.2e/%.2e" % (k, *v) for k, v in worst.items())))
    for k, (rb, fb) in BOUND.items():
        assert worst[k][0] <= rb, (k, "rounding oracle", worst[k][0], rb)
        assert worst[k][1] <= fb, (k, "float64 oracle", worst[k][1], fb)
    # the fused decay + Adam update: after three steps nearly every weight and bias equals the rounding oracle's to
    # within ADAM_ATOL (the rest are elements whose tiny gradients changed sign).  The same check against oracles
    # without the decay or with a 10 % larger step size must fail: it sees a wrong update.
    got = [np.concatenate([t.cpu().numpy().ravel() for t in engine.get_weights(which, l)]) for l in range(nl)]

    def close(Wb):
        return min(float(np.mean(np.abs(g - np.concatenate([Wb[0][l].ravel(), Wb[1][l].ravel()])) <= ADAM_ATOL))
                   for l, g in enumerate(got))

    def wrong(decay_, lr_):
        opt = tro.Adam([p for l in range(nl) for p in (W[l], b[l])], lr=lr_)
        st = (W, b)
        for _ in range(3):
            r = trb.train_step(*st, ens.acts, x64, y64, loss, opt, decay_, round_bf16=True, **sc)
            st = (r[1], r[2])
        return st

    frac = close(state[0])
    frac_bad = max(close(wrong(0.0, 1e-3)), close(wrong(decay, 1.1e-3)))
    print("bf16 Adam %s: fraction within %.0e: %.4f (wrong update: %.4f)" % (name, ADAM_ATOL, frac, frac_bad))
    assert frac >= ADAM_FRAC, (frac, ADAM_FRAC)
    assert frac_bad < ADAM_FRAC, frac_bad


def _snapshot(engine, which, nl, lout):
    out = [lout.cpu().numpy().copy()]
    for l in range(nl):
        out += [t.cpu().numpy().copy() for t in engine.get_weights(which, l) + engine.train_grads(which, l)]
    return out


@pytest.mark.parametrize("name", ["hcs", "humanoid", "e8_bs257_tanh"])
def test_bf16_steps_are_deterministic(engine, name):
    runs = []
    for _ in range(2):
        model, ens, which, x, y, loss = _case(engine, name)
        model.configure_training(loss=loss, math="bf16")
        engine.train_begin(which)
        lout = engine.empty(ens.W[0].shape[0])
        snaps = []
        for _ in range(3):
            engine.train_step(which, x, y, model._train_cfg, lout)
            snaps.append(_snapshot(engine, which, len(ens.W), lout))
        runs.append(snaps)
    for s0, s1 in zip(*runs):
        for a, b in zip(s0, s1):
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.parametrize("name", ["hcs", "v_mse"])
def test_w16_follows_fp32_and_tf32_steps(engine, name):
    """fp32, bf16, TF32, bf16 on one optimiser state.  Every step's loss and gradients match its own mode's oracle
    evaluated at the weights the device holds before the step, so each bf16 step reads weights that include the
    update of the step before (a stale W16 would miss a whole Adam step of lr = 1e-2)."""
    model, ens, which, x, y, loss = _case(engine, name)
    _, _, sc = _f64(ens)
    nl = len(ens.W)
    x64, y64 = x.astype(np.float64), y.astype(np.float64)
    lout = engine.empty(ens.W[0].shape[0])
    engine.train_begin(which)
    for math in ("fp32", "bf16", "tf32", "bf16"):
        model.configure_training(loss=loss, lr=1e-2, decay=1e-2, math=math)
        wb = [engine.get_weights(which, l) for l in range(nl)]
        W = [w.cpu().numpy().astype(np.float64) for w, _ in wb]
        b = [bb.cpu().numpy().astype(np.float64) for _, bb in wb]
        if math == "bf16":
            want = trb.grads(W, b, ens.acts, x64, y64, loss, round_bf16=True, **sc)
            ltol, gtol = BOUND["loss"][1], max(BOUND["dW"][1], BOUND["db"][1])
        else:
            want = tro.grads(W, b, ens.acts, x64, y64, loss, **sc)
            ltol, gtol = OTHER[math]
        engine.train_step(which, x, y, model._train_cfg, lout)
        assert _loss_rel(lout.cpu().numpy(), want[0]) <= ltol, (math, _loss_rel(lout.cpu().numpy(), want[0]))
        for l in range(nl):
            dW, db = (t.cpu().numpy() for t in engine.train_grads(which, l))
            assert _rel(dW, want[1][l]) <= gtol, (math, "dW", l, _rel(dW, want[1][l]))
            assert _rel(db, want[2][l]) <= gtol, (math, "db", l, _rel(db, want[2][l]))


@pytest.mark.parametrize("name", ["hcs", "humanoid"])
def test_bf16_step_launch_count(engine, name):
    """3L + 2 launches per bf16 step; L more on a step that rebuilds W16 (new state, or after an fp32 step)."""
    model, ens, which, x, y, loss = _case(engine, name)
    L = len(ens.W)
    engine.train_begin(which)
    x, y = engine.to_device(x, engine.torch.float32), engine.to_device(y, engine.torch.float32)

    def launches(math):
        model.configure_training(loss=loss, math=math)
        n0 = engine.launch_count
        engine.train_step(which, x, y, model._train_cfg)
        return engine.launch_count - n0

    assert launches("bf16") == 4 * L + 2
    assert launches("bf16") == 3 * L + 2
    assert launches("bf16") == 3 * L + 2
    launches("fp32")
    assert launches("bf16") == 4 * L + 2
    assert launches("bf16") == 3 * L + 2


def test_train_loop_learns_and_repacks_bf16(engine):
    """B200PE.train with math='bf16' meets the bounds of test_gpu_train.py::test_train_loop_learns_and_repacks."""
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    O, A, E = 17, 6, 7
    rng = np.random.RandomState(0)
    dyn, _, _, _ = orc.make_problem(21, O, A, hidden=(128, 128), num_nets=E, num_elites=5, gain=1.0)
    model = cb.B200PE.from_arrays(engine, L.NET_DYN, dyn)
    n = 4096
    X = rng.standard_normal((n, O + A)).astype(np.float32)
    M = (rng.standard_normal((O + A, O + 1)) * 0.3).astype(np.float32)
    Y = (np.tanh(X @ M) + 0.05 * rng.standard_normal((n, O + 1))).astype(np.float32)
    model.configure_training(loss="MSPE", lr=1e-3, decay=1e-6, use_scaler_in=True, use_scaler_out=True, math="bf16")
    before = model.validate(X[:512], Y[:512])
    out = model.train(X, Y, batch_size=256, max_epochs=15, holdout_ratio=0.1, rng=rng)
    after = model.validate(X[:512], Y[:512])
    assert after < 0.35 * before, (before, after)
    assert list(out.keys()) == ["PE/val_loss"] and np.isfinite(out["PE/val_loss"])
    assert len(model.elite_inds) == 5 and len(set(model.elite_inds)) == 5
    assert model._grad_updates == 15 * int(np.ceil((n - 409) / 256))
    m16, v16 = model.predict_ensemble_device(X[:1000], precision="fp16")
    m32, v32 = model.predict_ensemble_device(X[:1000], precision="fp32")
    np.testing.assert_allclose(m16.cpu().numpy(), m32.cpu().numpy(), rtol=2e-2, atol=2e-2)
    assert engine.nets[L.NET_DYN]["elite_inds"] == model.elite_inds


def test_unknown_math_is_rejected(engine):
    from cmbpo_b200 import _lib as L
    model, ens, which, x, y, loss = _case(engine, "v_mse")
    for bad in ("fp16", "TF32", "", None, 2):
        with pytest.raises(ValueError):
            model.configure_training(loss=loss, math=bad)
    model.configure_training(loss=loss, math="bf16")
    engine.train_begin(which)
    W0 = engine.get_weights(which, 0)[0].cpu().numpy()
    cfg = model._train_cfg
    for bad in (3, -1, 100):
        cfg.math = bad
        with pytest.raises(L.CmbpoError, match="math"):
            engine.train_step(which, x, y, cfg)
    assert np.array_equal(engine.get_weights(which, 0)[0].cpu().numpy(), W0)
