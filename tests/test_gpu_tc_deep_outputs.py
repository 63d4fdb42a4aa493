"""Deep dynamics ensembles (3 or 4 hidden layers, padded width 256) with 65 to 128 output columns on the tensor cores:
the wide-output deep kernels of csrc/ens_tc.cu (WO), e.g. a probabilistic HumanoidSafe model with the reference's
code-default architecture (200, 200, 200, 200) (algorithms/cmbpo.py:54): 2 x (47 observations + reward) = 96 outputs.

K1 is checked against the two float64 references and bounds of test_gpu_tc_variants.py, restated here:
  * `forward64`: the operation itself, float64 end to end; mean error at most 1 unit of 1e-3 |want| + 1e-3 sigma_out
    for fp16 and 8 units for bf16, variance relative error at most 1e-3 / 1e-2;
  * `forward64_q`: float64 that rounds where the kernel rounds; at most about twice the residual measured there.
Every network has non-zero biases in every layer.
"""
import zlib

import numpy as np
import pytest

from helpers import TASKS, GAE, ShapeEnv, calibrated_dkl_lim, load_problem
from oracle import cmbpo_oracle as orc

pytestmark = pytest.mark.gpu

F32, F64 = np.float32, np.float64
SCALE = {"fp16": 1.0, "bf16": 8.0}
VTOL = {"fp16": 1e-3, "bf16": 1e-2}
Q_BOUND = {"fp16": 0.2, "bf16": 1.5}
Q_VTOL = {"fp16": 2.7e-4, "bf16": 1.7e-3}
SIGNED_BOUND = 0.3


@pytest.fixture(scope="module")
def eng():
    """A context of its own: the networks loaded here do not outlive this module."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    import cmbpo_b200
    e = cmbpo_b200.Engine(0, precision="fp32")
    yield e
    e.close()


# ---------------------------------------------------------------------------------------------------- references
def _sig64(var):
    return np.maximum(np.sqrt(np.asarray(var, F64).reshape(-1)), 1e-2)


def _sig32(var):
    return np.maximum(np.sqrt(np.asarray(var, F32).reshape(-1)), F32(1e-2))


def _head64(ens, raw):
    """output scaler and exp(logvar) (pe.py:789-838) on the raw last-layer output [E, N, out]"""
    D = ens.out_dim
    sig = _sig64(ens.var_out)
    mean = sig * raw[..., :D] + np.asarray(ens.mu_out, F64).reshape(-1)
    if not ens.probabilistic:
        return mean, None
    with np.errstate(over="ignore"):
        return mean, np.exp(2.0 * np.log(sig) + raw[..., D:])


def forward64(ens, x):
    h = (np.asarray(x, F64) - np.asarray(ens.mu_in, F64).reshape(-1)) / _sig64(ens.var_in)
    for W, b, a in zip(ens.W, ens.b, ens.acts):
        h = np.matmul(h, np.asarray(W, F64)) + np.asarray(b, F64).reshape(W.shape[0], 1, -1)
        if a == "swish":
            with np.errstate(over="ignore"):
                h = h / (1.0 + np.exp(-h))
        elif a == "tanh":
            h = np.tanh(h)
    return _head64(ens, h)


def _q16(a, fmt):
    """float32 -> fp16 (saturating) or bf16, round to nearest even, back to float64"""
    a = np.asarray(a, F32)
    if fmt == "fp16":
        return np.clip(a, -65504, 65504).astype(np.float16).astype(F64)
    u = a.view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(F32).astype(F64)


def forward64_q(ens, x, fmt):
    """forward64 with the kernel's 16-bit rounding points: scaled inputs, weights (swish layers pre-halved), the
    layer-0 bias as a hi / lo pair when it rides in the GEMM (K0 + 2 <= 64), hidden activations."""
    E, K0 = ens.W[0].shape[:2]
    swish = ens.acts[0] == "swish"
    half = F32(0.5) if swish else F32(1.0)
    z = (np.asarray(x, F32) - np.asarray(ens.mu_in, F32).reshape(-1)).astype(F32) / _sig32(ens.var_in)
    h = _q16(z, fmt)
    L = len(ens.W)
    for l in range(L):
        s = F32(1.0) if l == L - 1 else half
        Wq = _q16(np.asarray(ens.W[l], F32) * s, fmt)
        bl = (np.asarray(ens.b[l], F32).reshape(E, 1, -1) * s).astype(F32)
        if l == 0 and K0 + 2 <= 64:
            hi = _q16(bl, fmt)
            bias = hi + _q16(bl - hi.astype(F32), fmt)
        else:
            bias = bl.astype(F64)
        t = np.matmul(h, Wq) + bias
        if l == L - 1:
            return _head64(ens, t)
        h = _q16(t + t * np.tanh(t) if swish else np.tanh(t), fmt)


def _units(got, want, sig):
    """max error in units of the stated tolerance 1e-3 |want| + 1e-3 sigma_out"""
    return float(np.max(np.abs(got - want) / (1e-3 * np.abs(want) + 1e-3 * sig)))


def _vrel(got, want):
    return float(np.max(np.abs(got - want) / want))


def _signed(got, want, sig):
    """max over output columns of |mean signed error| / RMS error (an RMS below 0.01 units counts as 0.01)"""
    d = ((np.asarray(got, F64) - want) / (1e-3 * np.abs(want) + 1e-3 * sig)).reshape(-1, got.shape[-1])
    rms = np.maximum(np.sqrt(np.mean(d * d, axis=0)), 0.01)
    return float(np.max(np.abs(d.mean(axis=0)) / rms))


def _ensemble(seed, K0, hidden, D, prob, act, E):
    """fc.py-scale weights, non-zero biases in every layer, data-like input / output scalers"""
    rng = np.random.default_rng(seed)
    s = np.exp(rng.uniform(np.log(0.05), np.log(3.0), K0))
    so = np.exp(rng.uniform(np.log(0.05), np.log(2.0), D))
    scalers = (rng.standard_normal(K0) * s, s ** 2, 0.1 * rng.standard_normal(D), so ** 2)
    ens = orc.make_ensemble(rng, K0, D, hidden, E, max(1, E - 2), prob, act=act, scalers=scalers, gain=1.0,
                            bias_std=rng.uniform(0.1, 0.5))
    return ens, rng


def _rows(rng, ens, N):
    mu, var = ens.mu_in.reshape(-1).astype(F64), ens.var_in.reshape(-1).astype(F64)
    return (mu + _sig64(var) * rng.standard_normal((N, mu.size))).astype(F32)


# ---------------------------------------------------------------------------------------------------- K1
# (id, inputs K0, hidden widths, outputs D (x2 when probabilistic), probabilistic, activation, members E, rows N)
CASES = [
    ("d4_swish_out96_hum", 64, (200,) * 4, 48, True, "swish", 7, 38145),
    ("d3_swish_out96_hum_E1", 64, (200,) * 3, 48, True, "swish", 1, 129),
    ("d3_tanh_out96_w128", 64, (128,) * 3, 48, True, "tanh", 7, 127),
    ("d3_swish_out65", 20, (200,) * 3, 65, False, "swish", 7, 1000),
    ("d4_tanh_out65_w128_E1", 23, (128,) * 4, 65, False, "tanh", 1, 127),
    ("d3_swish_out97_w128", 17, (128,) * 3, 97, False, "swish", 7, 1),
    ("d4_tanh_out97", 20, (200,) * 4, 97, False, "tanh", 7, 129),
    ("d3_tanh_out128_prob", 20, (200,) * 3, 64, True, "tanh", 7, 38145),
    ("d4_swish_out128_w128_E1", 20, (128,) * 4, 128, False, "swish", 1, 1),
    ("d4_swish_out128_prob_w256", 30, (256,) * 4, 64, True, "swish", 7, 127),
    ("d4_tanh_out128_E1", 40, (200,) * 4, 128, False, "tanh", 1, 38145),
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_deep_wide_output_vs_float64(eng, case):
    """predict_ensemble and predict_mean at fp16 and bf16 against forward64 (stated rule) and forward64_q (tight
    bound, unbiased residual); the first rows of the batch give the same bits when run alone."""
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    name, K0, hidden, D, prob, act, E, N = case
    ens, rng = _ensemble(zlib.crc32(name.encode()), K0, hidden, D, prob, act, E)
    model = cb.B200PE.from_arrays(eng, L.NET_DYN, ens)
    x = _rows(rng, ens, N)
    sel = np.arange(N) if N <= 2000 else np.unique(np.concatenate([np.arange(300), np.arange(N - 300, N),
                                                                  rng.choice(N, 400, replace=False)]))
    wm, wv = forward64(ens, x[sel])
    sig = _sig64(ens.var_out)
    R = min(N - 1, 200)
    for fmt in ("fp16", "bf16"):
        out = model.predict_ensemble_device(x, precision=fmt)
        gm, gv = (t.cpu().numpy() for t in out) if prob else (out.cpu().numpy(), None)
        assert gm.shape == (E, N, D) and np.isfinite(gm).all()
        gm = gm[:, sel]
        qm, qv = forward64_q(ens, x[sel], fmt)
        e64, eq, sg = _units(gm, wm, sig), _units(gm, qm, sig), _signed(gm, qm, sig)
        msg = "%s %s: float64 %.3f units" % (name, fmt, e64)
        if prob:
            gv = gv[:, sel]
            v64, vq = _vrel(gv, wv), _vrel(gv, qv)
            msg += " var %.2e" % v64
        msg += " | 16-bit ref %.3f units" % eq + (" var %.2e" % vq if prob else "") + " | signed %.3f" % sg
        pm = model.predict_device(x, precision=fmt)
        pm, pv = (t.cpu().numpy() for t in pm) if prob else (pm.cpu().numpy(), None)
        mm = wm.mean(axis=0)
        em = _units(pm[sel], mm, sig)
        msg += " | mean of members %.3f units" % em
        print(msg)
        assert e64 <= SCALE[fmt], msg
        assert em <= SCALE[fmt], msg
        assert eq <= Q_BOUND[fmt], msg
        if gm.size >= 2000:
            assert sg <= SIGNED_BOUND, msg
        if prob:
            assert v64 <= VTOL[fmt], msg
            assert vq <= Q_VTOL[fmt], msg
            wpv = wv.mean(axis=0) + np.mean(np.square(wm - mm), axis=0)
            assert _vrel(pv[sel], wpv) <= VTOL[fmt], msg
        if R >= 1:                                    # row r depends on row r only
            sub = model.predict_ensemble_device(x[:R], precision=fmt)
            full = model.predict_ensemble_device(x, precision=fmt)
            for a, b in zip(sub if prob else (sub,), full if prob else (full,)):
                assert np.array_equal(a.cpu().numpy(), b.cpu().numpy()[:, :R]), name


@pytest.mark.parametrize("layers", [3, 4])
def test_deep_wide_output_many_units(eng, layers):
    """E = 7 and 20 000 rows: about seven work units per CTA, so the last hidden buffer, the OUT accumulator and the
    per-chunk hand-off barriers go through many phases in one launch.  Checked against the fp32 path."""
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    task, O, A = TASKS["hum"]
    dyn, actor, v, vc = orc.make_problem(101 + layers, O, A, hidden=(200,) * layers, task=task)
    rb = np.random.default_rng(100 + layers)
    for bl in dyn.b:
        bl += (0.1 * rb.standard_normal(bl.shape)).astype(F32)
    model = cb.B200PE.from_arrays(eng, L.NET_DYN, dyn)
    obs, act = orc.make_states(102, 20000, O, A, dyn)
    x = eng.to_device(np.concatenate([obs, act], -1))
    m32, v32 = model.predict_ensemble_device(x, precision="fp32")
    m16, v16 = model.predict_ensemble_device(x, precision="fp16")
    eng.synchronize()
    assert m16.shape == (7, 20000, O + 1)
    assert bool(m16.isfinite().all()) and bool(v16.isfinite().all())
    sig = eng.to_device(_sig64(dyn.var_out).astype(F32))
    err = float(((m16 - m32).abs() / (1e-3 * m32.abs() + 1e-3 * sig)).max())
    verr = float(((v16 - v32).abs() / v32).max())
    print("deep %d layers, 96 outputs, 20000 rows: mean %.3f units, var %.2e" % (layers, err, verr))
    assert err <= 1.0 and verr <= 1.5e-3, (err, verr)


# ---------------------------------------------------------------------------------------------------- rollout
def _hum_deep_problem(seed):
    task, O, A = TASKS["hum"]
    dyn, actor, v, vc = orc.make_problem(seed, O, A, hidden=(200, 200, 200, 200), task=task)
    rb = np.random.default_rng(seed + 1)
    for bl in dyn.b:
        bl += (0.1 * rb.standard_normal(bl.shape)).astype(F32)
    return task, O, A, dyn, actor, v, vc


def test_rollout_humanoid_deep_fp16_vs_fp32(eng):
    """The HumanoidSafe code-default model: single-step prediction against the oracle and a short rollout at fp16
    against the fp32 CUDA-core path, with the checks of test_rollout_tc_padded_widths_and_real_hcs_obs."""
    import cmbpo_b200 as cb
    task, O, A, dyn, actor, v, vc = _hum_deep_problem(111)
    B, T = 700, 6
    obs, act = orc.make_states(112, B, O, A, dyn)
    model, policy = load_problem(eng, dyn, actor, v, vc)
    x = np.concatenate([obs, act], axis=1)
    want_m, want_v = orc.pe_forward(dyn, x)
    got_m, got_v = (t.cpu().numpy() for t in model.predict_ensemble_device(x, precision="fp16"))
    sig = _sig64(dyn.var_out)
    assert _units(got_m, want_m, sig) <= 1.0
    assert float(np.max(np.abs(got_v - want_v) / want_v)) <= 1.5e-3
    noise = orc.TableNoise(113, T, B, A, len(dyn.elite_inds))
    env = cb.FakeEnv(ShapeEnv(O, A), task, model, True, True, False)
    res = {}
    for prec in ("fp32", "fp16"):
        bufs = cb.RolloutBuffers(eng, B, T, O, A)
        bufs.set_inputs(obs, noise.act_eps, noise.elite_pos)
        bufs.run(env.env_cfg(True), precision=prec)
        eng.synchronize()
        res[prec] = bufs
    a, b = res["fp32"], res["fp16"]
    la, lb = a.length.cpu().numpy(), b.length.cpu().numpy()
    assert (la != lb).mean() <= 0.02 + 1.0 / B
    same = la == lb
    scale = np.maximum(np.sqrt(dyn.var_in[0, :O]), 1e-2)
    na, nb = a.host("nextobs"), b.host("nextobs")
    va, vb = a.host("val"), b.host("val")
    checked = 0
    for t in range(T - 1):
        m = same & (la > t)
        if m.any():
            checked += 1
            assert np.max(np.abs(na[m, t] - nb[m, t]) / scale) <= 3e-3 * (t + 1), t
            assert np.allclose(va[m, t], vb[m, t], rtol=2e-2, atol=2e-2), t
    assert checked == T - 1


def test_rollout_humanoid_deep_compaction_is_invisible(eng):
    """Uncertainty mode (paths cut at a cumulative-KL limit) with the deep 96-output model at fp16: squeezing the
    finished paths out of the batch changes no bit of any output."""
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    task, O, A, dyn, actor, v, vc = _hum_deep_problem(121)
    B, T = 6000, 35
    load_problem(eng, dyn, actor, v, vc)
    obs, act = orc.make_states(122, B, O, A, dyn)
    lim = calibrated_dkl_lim(dyn, task, obs[:2000], act[:2000], factor=10.0)
    cfg = L.EnvCfg(L.TERM_NO_DONE, L.COST_ZERO, 0, 1, 1)
    t = eng.torch
    res = []
    for flags in (0, L.ROLLOUT_NO_COMPACT):
        bufs = cb.RolloutBuffers(eng, B, T, O, A)
        bufs.set_inputs(obs)
        bufs.run(cfg, uncertainty_mode=True, dkl_lim=lim, seed=23, precision="fp16", flags=flags)
        bufs.gae(GAE["gamma"], GAE["lam"], GAE["cost_gamma"], GAE["cost_lam"])
        eng.synchronize()
        res.append(bufs)
    a, b = res
    ln = a.length.cpu().numpy()
    print("path lengths: mean %.1f, %d distinct" % (ln.mean(), len(np.unique(ln))))
    assert ln.mean() < T - 3 and len(np.unique(ln)) >= 3      # paths really end, at different steps
    for name in ("length", "end_reason", "last_val", "last_cval", "obs", "nextobs", "act", "mu", "rew", "val", "cval",
                 "logp", "cost", "dkl", "dyn_error", "term", "adv", "ret", "cadv", "cret", "cum_dkl"):
        assert bool(t.equal(getattr(a, name), getattr(b, name))), name


# ---------------------------------------------------------------------------------------------------- training
def test_training_repacks_the_deep_wide_output_model(eng):
    """B200PE.train on a deep 96-output model: train_end packs the trained weights again, so the fp16 / bf16
    predictions follow the fp32 ones afterwards.  (A small learning rate keeps the trained weights near the fc.py
    scale the stated tolerance is defined at: Adam moves every weight by about lr per step.)"""
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    ens, rng = _ensemble(131, 64, (200,) * 4, 48, True, "swish", 7)
    model = cb.B200PE.from_arrays(eng, L.NET_DYN, ens)
    x = _rows(rng, ens, 3000)
    before = model.predict_device(x, precision="fp16")[0].cpu().numpy()
    X = _rows(rng, ens, 4096)
    M = (rng.standard_normal((64, 48)) * 0.3).astype(F32)
    Xs = ((X - ens.mu_in.reshape(-1)) / _sig64(ens.var_in)).astype(F32)
    Y = (np.tanh(Xs @ M) + 0.05 * rng.standard_normal((4096, 48))).astype(F32)
    model.configure_training(loss="MSPE", lr=1e-4, use_scaler_in=True)
    model.train(X, Y, batch_size=256, max_epochs=2, holdout_ratio=0.1, hide_progress=True, rng=np.random.RandomState(132))
    ref, ref_v = (t.cpu().numpy() for t in model.predict_ensemble_device(x, precision="fp32"))
    sig = _sig64(ens.var_out)
    moved = _units(model.predict_device(x, precision="fp16")[0].cpu().numpy(), before, sig)
    print("fp16 member mean moved by %.1f units in training" % moved)
    assert moved > 10.0
    for fmt in ("fp16", "bf16"):
        got, got_v = (t.cpu().numpy() for t in model.predict_ensemble_device(x, precision=fmt))
        e, ev = _units(got, ref, sig), _vrel(got_v, ref_v)
        print("trained deep 96-output model %s: %.3f units, var %.2e against fp32" % (fmt, e, ev))
        assert e <= SCALE[fmt] and ev <= VTOL[fmt], (fmt, e, ev)


# ---------------------------------------------------------------------------------------------------- still rejected
@pytest.mark.parametrize("hidden,D,prob", [((200,) * 4, 65, True), ((200,) * 3, 129, False), ((512,) * 3, 48, True)],
                         ids=["deep_out130", "deep_out129", "deep_w512"])
def test_deep_shapes_beyond_the_limits_name_fp32(eng, hidden, D, prob):
    """More than 128 outputs, or a deep net wider than 256: an error naming fp32 on the tensor cores; fp32 works."""
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    ens, rng = _ensemble(141, 20, hidden, D, prob, "swish", 3)
    model = cb.B200PE.from_arrays(eng, L.NET_DYN, ens)
    x = _rows(rng, ens, 50)
    for fmt in ("fp16", "bf16"):
        with pytest.raises(cb.CmbpoError, match="fp32"):
            model.predict_ensemble_device(x, precision=fmt)
            eng.synchronize()
    out = model.predict_ensemble_device(x, precision="fp32")
    m = (out[0] if prob else out).cpu().numpy()
    assert _units(m, forward64(ens, x)[0], _sig64(ens.var_out)) <= 1.0
