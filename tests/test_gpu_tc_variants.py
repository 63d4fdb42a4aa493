"""Every tcgen05 kernel variant (csrc/ens_tc.cu: width 128 / 256 / 512, swish / tanh / per-member activation,
cluster pairs, grouped 4 x 128 units, the deep variants, the bias fold and the two-part output) and the tensor-core
policy pass against a float64 reference, with non-zero biases in every layer.

Two references:
  * `forward64` / `policy64`: the operation itself (pe.py / fc.py as the oracle cites them) in float64 end to end.
    Checked with the rule of test_gpu_tc.py, not loosened for any variant: mean error at most 1 unit of
    1e-3 |want| + 1e-3 sigma_out for fp16 and 8 units for bf16; variance relative error at most 1e-3 / 1e-2.
  * `forward64_q` / `policy64_q`: float64 that rounds where the kernel rounds (scaled inputs, weights with swish layers
    pre-halved, the layer-0 bias as a hi / lo pair when it rides in the GEMM, hidden activations; the merged policy
    pack's first layer folded in fp32 / float64 first).  What remains is tanh.approx.f32 and the fp32 accumulation
    order, so the bounds are tight.  Measured over this whole file on a B200 (1000 W power limit), worst ratio:
      - K1 against forward64_q: fp16 0.106, bf16 0.769 units; variance 1.3e-4 / 8.3e-4 (Q_BOUND, Q_VTOL: about 2x);
      - policy pass against policy64_q: fp16 0.190, bf16 1.70 units (Q_BOUND_POLICY: about 2x);
      - against forward64 / policy64: K1 fp16 0.26, bf16 2.1 units; policy fp16 0.55, bf16 3.7 units.
    The mean signed residual of every output column against forward64_q is also held small against its RMS
    (SIGNED_BOUND; measured at most 0.15): a conversion that truncates instead of rounding to nearest measured 0.81.
    Weights are at the scale of the fc.py initialiser (orc.make_ensemble gain 1).
"""
import zlib

import numpy as np
import pytest

from oracle import cmbpo_oracle as orc

pytestmark = pytest.mark.gpu

F32, F64 = np.float32, np.float64
SCALE = {"fp16": 1.0, "bf16": 8.0}             # units of the stated tolerance, test_gpu_tc.py
VTOL = {"fp16": 1e-3, "bf16": 1e-2}
Q_BOUND = {"fp16": 0.2, "bf16": 1.5}          # K1 against forward64_q, same units
Q_BOUND_POLICY = {"fp16": 0.4, "bf16": 3.4}   # policy pass against policy64_q
Q_VTOL = {"fp16": 2.7e-4, "bf16": 1.7e-3}     # variance relative error against forward64_q
SIGNED_BOUND = 0.3                             # |mean signed residual| / RMS residual, per output column


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
    """the device's sigma: max(sqrtf(var), 1e-2f) in float32 (train.cu prep_scaler2_kernel)"""
    return np.maximum(np.sqrt(np.asarray(var, F32).reshape(-1)), F32(1e-2))


def _act64(a, x):
    if a is None:
        return x
    if a == "swish":
        with np.errstate(over="ignore"):
            return x / (1.0 + np.exp(-x))
    if a == "tanh":
        return np.tanh(x)
    if a == "ReLU":
        return np.maximum(x, 0.0)
    raise ValueError(a)


def _head64(ens, raw):
    """output scaler and exp(logvar) (pe.py:789-838) on the raw last-layer output [E, N, out]"""
    D = ens.out_dim
    mean, var = raw[..., :D], None
    sig = _sig64(ens.var_out) if ens.mu_out is not None else None
    if sig is not None:
        mean = sig * mean + np.asarray(ens.mu_out, F64).reshape(-1)
    if ens.probabilistic:
        logvar = raw[..., D:]
        if sig is not None:
            logvar = 2.0 * np.log(sig) + logvar
        with np.errstate(over="ignore"):
            var = np.exp(logvar)
    return mean, var


def forward64(ens, x):
    """PE forward of every member on 2-D rows x, float64 end to end: (mean, var or None), each [E, N, D]."""
    h = np.asarray(x, F64)
    if ens.mu_in is not None:
        h = (h - np.asarray(ens.mu_in, F64).reshape(-1)) / _sig64(ens.var_in)
    for W, b, a in zip(ens.W, ens.b, ens.acts):
        h = _act64(a, np.matmul(h, np.asarray(W, F64)) + np.asarray(b, F64).reshape(W.shape[0], 1, -1))
    return _head64(ens, h)


def _q16(a, fmt):
    """float32 -> fp16 (saturating at +-65504) or bf16, round to nearest even, back to float64"""
    a = np.asarray(a, F32)
    if fmt == "fp16":
        return np.clip(a, -65504, 65504).astype(np.float16).astype(F64)
    u = a.view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(F32).astype(F64)


def _chain_q(z, W, b, member_acts, fmt):
    """the kernel's GEMM chain on scaled fp32 inputs z [N, K0]: W[l] [E, in, out], b[l] [E, out] (fp32),
    member_acts[e] = 'swish' | 'tanh'.  Returns the raw last-layer output [E, N, out] in float64."""
    E, K0 = W[0].shape[:2]
    swish = np.array([a == "swish" for a in member_acts]).reshape(E, 1, 1)
    half = np.where(swish, F32(0.5), F32(1.0)).astype(F32)       # ens_tc.cu:853-858: swish layers pre-halved
    h = _q16(z, fmt)
    L = len(W)
    for l in range(L):
        s = F32(1.0) if l == L - 1 else half
        Wq = _q16(np.asarray(W[l], F32) * s, fmt)
        bl = (np.asarray(b[l], F32).reshape(E, 1, -1) * s).astype(F32)
        if l == 0 and K0 + 2 <= 64:                               # bias rides in the GEMM as a (hi, lo) pair
            hi = _q16(bl, fmt)
            bias = hi + _q16(bl - hi.astype(F32), fmt)
        else:
            bias = bl.astype(F64)
        t = np.matmul(h, Wq) + bias
        if l == L - 1:
            return t
        with np.errstate(over="ignore"):
            h = _q16(np.where(swish, t + t * np.tanh(t), np.tanh(t)), fmt)   # swish(2t) = t + t tanh t


def _scale32(ens, x):
    x = np.asarray(x, F32)
    if ens.mu_in is None:
        return x
    return (x - np.asarray(ens.mu_in, F32).reshape(-1)).astype(F32) / _sig32(ens.var_in)


def forward64_q(ens, x, fmt):
    """forward64 with the kernel's 16-bit rounding points (fmt = 'fp16' | 'bf16')."""
    E = ens.num_nets
    raw = _chain_q(_scale32(ens, x), ens.W, [b.reshape(E, -1) for b in ens.b], [ens.acts[0]] * E, fmt)
    return _head64(ens, raw)


def _actor_ens(actor):
    return orc.Ensemble([w[None] for w in actor.W], [b.reshape(1, 1, -1) for b in actor.b],
                        ["tanh"] * (len(actor.W) - 1) + [None], False)


def _values64(ens, obs, fwd):
    return fwd(ens, obs)[0][..., 0].mean(axis=0)


def policy64(actor, v, vc, obs, eps):
    """actor mu, pi = mu + eps exp(log_std), logp (ac_network.py:46-48, 109), v / vc = member means (pe.py:648-669)"""
    mu = forward64(_actor_ens(actor), obs)[0][0]
    ls = np.asarray(actor.log_std, F64)
    pi = mu + np.asarray(eps, F64) * np.exp(ls)
    return dict(mu=mu, pi=pi, logp=_logp64(pi, mu, ls),
                v=_values64(v, obs, forward64), vc=_values64(vc, obs, forward64))


def _logp64(pi, mu, ls):
    z = (pi - mu) / (np.exp(ls) + orc.LOGP_EPS)
    return -0.5 * np.sum(z * z + 2.0 * ls + np.log(2 * np.pi), axis=1)


def _tc_ok(ens):
    """ens_tc_supported (ens_tc.cu:1062-1071)"""
    dims = [ens.W[0].shape[1]] + [w.shape[2] for w in ens.W]
    L = len(ens.W)
    if L < 3 or L > 5 or any(d != dims[1] for d in dims[1:L]) or dims[1] > (512 if L == 3 else 256):
        return False
    if dims[0] > 64 or dims[L] > ((96 if dims[1] > 256 else 128) if L == 3 else 64):
        return False
    return all(a == ens.acts[0] for a in ens.acts[:-1]) and ens.acts[-1] is None and ens.acts[0] in ("swish", "tanh")


def _merged(actor_e, v, vc):
    """policy_pack_build's conditions (policy_pack.cu:46-67)"""
    hd, O = actor_e.W[0].shape[2], actor_e.W[0].shape[1]

    def ok(n):
        return (len(n.W) == 3 and n.W[0].shape[1] == O and n.W[0].shape[2] == hd and n.W[1].shape[2] == hd
                and n.acts[0] == n.acts[1] and n.acts[0] in ("swish", "tanh") and not n.probabilistic)
    return (hd in (128, 256) and ok(actor_e) and ok(v) and ok(vc) and v.out_dim == 1 and vc.out_dim == 1 and O <= 64
            and 1 + v.num_nets + vc.num_nets <= 8)


def policy64_q(actor, v, vc, obs, fmt):
    """mu, v, vc with the rounding of the tensor-core policy pass: the merged pack when policy_pack_build builds one,
    else the three nets on their own (a net the tensor cores do not take runs in fp32: float64 stands for it)."""
    ae = _actor_ens(actor)
    if not _merged(ae, v, vc):
        def one(n):
            return forward64_q(n, obs, fmt) if _tc_ok(n) else forward64(n, obs)
        return dict(mu=one(ae)[0][0], v=one(v)[0][..., 0].mean(0), vc=one(vc)[0][..., 0].mean(0))
    O, A = obs.shape[1], actor.W[-1].shape[1]
    c = np.zeros(O, F32) if v.mu_in is None else np.asarray(v.mu_in, F32).reshape(-1)
    s = np.ones(O, F32) if v.mu_in is None else _sig32(v.var_in)
    z = (np.asarray(obs, F32) - c).astype(F32) / s
    Ws, bs, acts = [[], [], []], [[], [], []], []
    members = [(ae, 0)] + [(v, e) for e in range(v.num_nets)] + [(vc, e) for e in range(vc.num_nets)]
    for n, e in members:
        mn = np.zeros(O, F32) if n.mu_in is None else np.asarray(n.mu_in, F32).reshape(-1)
        sn = np.ones(O, F32) if n.mu_in is None else _sig32(n.var_in)
        w0 = np.asarray(n.W[0][e], F32)
        # fold_first_layer_kernel (policy_pack.cu:19-33): W0' in fp32, b0' accumulated in float64
        Ws[0].append(w0 * (s / sn).astype(F32)[:, None])
        bs[0].append((np.asarray(n.b[0][e], F64).reshape(-1) + ((c - mn) / sn).astype(F32).astype(F64) @ w0.astype(F64)).astype(F32))
        Ws[1].append(n.W[1][e])
        bs[1].append(n.b[1][e].reshape(-1))
        w2 = np.zeros((n.W[2].shape[1], A), F32)
        b2 = np.zeros(A, F32)
        w2[:, :n.W[2].shape[2]] = n.W[2][e]
        b2[:n.W[2].shape[2]] = n.b[2][e].reshape(-1)
        Ws[2].append(w2)
        bs[2].append(b2)
        acts.append(n.acts[0])
    raw = _chain_q(z, [np.stack(w) for w in Ws], [np.stack(b) for b in bs], acts, fmt)
    nv = v.num_nets

    def value(n, r):
        return (_sig64(n.var_out) * r + np.asarray(n.mu_out, F64).reshape(-1) if n.mu_out is not None else r).mean(0)
    return dict(mu=raw[0], v=value(v, raw[1:1 + nv, :, 0]), vc=value(vc, raw[1 + nv:, :, 0]))


# ---------------------------------------------------------------------------------------------------- measures
def _units(got, want, sig):
    """max error in units of the stated tolerance 1e-3 |want| + 1e-3 sigma_out"""
    return float(np.max(np.abs(got - want) / (1e-3 * np.abs(want) + 1e-3 * sig)))


def _vrel(got, want):
    return float(np.max(np.abs(got - want) / want))


def _signed(got, want, sig):
    """max over output columns of |mean signed error| / RMS error (all members and rows of a column), the error in
    units of the tolerance; an RMS below 0.01 units counts as 0.01 (a residual that is practically zero has no sign
    worth testing)"""
    d = ((np.asarray(got, F64) - want) / (1e-3 * np.abs(want) + 1e-3 * sig)).reshape(-1, got.shape[-1])
    rms = np.maximum(np.sqrt(np.mean(d * d, axis=0)), 0.01)
    return float(np.max(np.abs(d.mean(axis=0)) / rms))


def _scalers(rng, K, D, flat=True):
    """data-like input scaler with per-dimension scale in [0.05, 3]; two dimensions (when K >= 4) with a variance of
    1e-6, below the 1e-4 the sigma clamp of pens/utils.py:156 turns into sigma = 1e-2; output scaler likewise."""
    s = np.exp(rng.uniform(np.log(0.05), np.log(3.0), K))
    mu = rng.standard_normal(K) * s
    var = s ** 2
    if flat and K >= 4:
        var[rng.choice(K, 2, replace=False)] = 1e-6
    so = np.exp(rng.uniform(np.log(0.05), np.log(2.0), D))
    return mu, var, 0.1 * rng.standard_normal(D), so ** 2


def _rows(rng, ens, N):
    mu, var = ens.mu_in.reshape(-1).astype(F64), ens.var_in.reshape(-1).astype(F64)
    return (mu + _sig64(var) * rng.standard_normal((N, mu.size))).astype(F32)


def _ensemble(seed, K0, hidden, D, prob, act, E):
    rng = np.random.default_rng(seed)
    # weights at the scale of the fc.py initialiser, where the fp16 error sits well inside the stated tolerance
    ens = orc.make_ensemble(rng, K0, D, hidden, E, max(1, E - 2), prob, act=act, scalers=_scalers(rng, K0, D),
                            gain=1.0, bias_std=rng.uniform(0.1, 0.5))
    return ens, rng


# ---------------------------------------------------------------------------------------------------- K1 matrix
# (id, inputs K0, hidden widths, outputs D, probabilistic, activation, members E, rows N)
CASES = [
    ("tanh128", 23, (128, 128), 18, True, "tanh", 7, 1000),
    ("tanh256", 23, (256, 256), 18, True, "tanh", 5, 700),
    ("tanh512_pairs", 23, (512, 512), 18, True, "tanh", 7, 1500),
    ("tanh512_single", 23, (512, 512), 18, True, "tanh", 7, 100),
    ("swish512_pairs", 23, (512, 512), 18, True, "swish", 7, 1500),
    ("tanh_deep3", 20, (200, 200, 200), 18, True, "tanh", 7, 500),
    ("tanh_deep4", 20, (256,) * 4, 10, True, "tanh", 5, 300),
    ("swish_deep3_w128", 20, (128,) * 3, 18, True, "swish", 3, 300),
    ("swish_deep4", 23, (200,) * 4, 32, False, "swish", 7, 400),
    ("grouped_E2_swish", 17, (128, 128), 1, False, "swish", 2, 700),
    ("grouped_E3_tanh_w100", 17, (100, 100), 4, True, "tanh", 3, 500),
    ("grouped_E4_swish", 29, (128, 128), 8, True, "swish", 4, 300),
    ("grouped_E5_tanh", 17, (128, 128), 1, False, "tanh", 5, 400),
    ("grouped_E8_swish", 47, (128, 128), 3, False, "swish", 8, 260),
] + [("k0_%d" % k, k, (256, 256), 5, True, "tanh" if k in (15, 63) else "swish", 3, 300)
     for k in (1, 15, 16, 17, 62, 63, 64)] + [
    ("out%d_%s" % (d * (2 if p else 1), "prob" if p else "det"), 20, (256, 256), d, p, "swish", 3, 300)
    for d, p in ((1, False), (1, True), (16, False), (17, False), (32, True), (65, False), (48, True), (128, False),
                 (64, True))] + [
    ("out96_prob_w512_tanh", 20, (512, 512), 48, True, "tanh", 3, 300),
] + [("hid_%d" % h, 20, (h, h), 9, True, "tanh" if h in (65, 257) else "swish", 3, 300)
     for h in (1, 65, 129, 257, 511)] + [
    ("E1_w512", 23, (512, 512), 18, True, "swish", 1, 500),
    ("E1_w128", 17, (128, 128), 1, False, "tanh", 1, 300),
    ("E8_w256_tanh", 23, (256, 256), 18, True, "tanh", 8, 300),
] + [("N_%d" % n, 23, (512, 512), 18, True, "swish", 7, n) for n in (1, 127, 128, 129, 128 * 298 + 1)]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_k1_variant_vs_float64(eng, case):
    """predict_ensemble and predict_mean of one kernel variant at fp16 and bf16 against forward64 (stated rule) and
    forward64_q (tight bound, unbiased residual); the first rows of the batch give the same bits when run alone."""
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    name, K0, hidden, D, prob, act, E, N = case
    ens, rng = _ensemble(zlib.crc32(name.encode()), K0, hidden, D, prob, act, E)
    model = cb.B200PE.from_arrays(eng, L.NET_DYN, ens)
    x = _rows(rng, ens, N)
    # the float64 references on a sample of rows (all of them up to 2000): both ends of the batch and random rows
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
        # the member mean (pe.py:648-669)
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
        # row r depends on row r only
        if R >= 1:
            sub = model.predict_ensemble_device(x[:R], precision=fmt)
            full = model.predict_ensemble_device(x, precision=fmt)
            for a, b in zip(sub if prob else (sub,), full if prob else (full,)):
                assert np.array_equal(a.cpu().numpy(), b.cpu().numpy()[:, :R]), name


# ---------------------------------------------------------------------------------------------------- policy pass
def _policy_problem(seed, O=17, A=6, a_hidden=(128, 128), hidden=(128, 128), v_act="swish", vc_act=None, nv=3, nvc=3,
                    vc_scaler="same"):
    """actor + V + VC with non-zero biases everywhere.  vc_scaler: 'same' (V's input scaler), 'own' (a different
    one) or None (no input scaler)."""
    rng = np.random.default_rng(seed)
    mu_o, var_o, _, _ = _scalers(rng, O, 1)
    # the actor sees raw observations, 16-bit on the tensor cores when it runs alone: moderate first-layer gains
    actor = orc.make_actor(rng, O, A, a_hidden, gain=0.7)
    sig = np.maximum(np.sqrt(var_o), 1.0)
    w0 = actor.W[0].astype(F64)
    actor.W[0] = (w0 / sig[:, None]).astype(F32)
    actor.b = [(b + 0.3 * rng.standard_normal(b.shape)).astype(F32) for b in actor.b]
    actor.b[0] = (actor.b[0] - (mu_o / sig) @ w0).astype(F32)
    actor.log_std = rng.uniform(-1.0, 0.2, A).astype(F32)
    v = orc.make_ensemble(rng, O, 1, hidden, nv, 2, False, act=v_act, scalers=(mu_o, var_o, [3.0], [25.0]),
                          bias_std=0.3)
    if vc_scaler == "own":
        mu_c = mu_o + 0.5 * np.sqrt(var_o) * rng.standard_normal(O)
        var_c = var_o * np.exp(rng.uniform(-1.0, 1.0, O))
    else:
        mu_c, var_c = mu_o, var_o
    vc = orc.make_ensemble(rng, O, 1, hidden, nvc, 2, False, act=vc_act or v_act, scalers=(mu_c, var_c, [1.0], [4.0]),
                           bias_std=0.3)
    if vc_scaler is None:
        vc.mu_in = vc.var_in = None
    obs = (mu_o + _sig64(var_o) * rng.standard_normal((777, O))).astype(F32)
    eps = rng.standard_normal((777, A)).astype(F32)
    return actor, v, vc, obs, eps


def _load_policy(eng, actor, v, vc):
    import cmbpo_b200 as cb
    policy = cb.B200Policy(eng)
    policy.load_actor(actor.W, actor.b, actor.log_std)
    policy.load_values(v, vc)
    return policy


def _check_policy(eng, actor, v, vc, obs, eps, fmt, label):
    """mu / v / vc against policy64 (stated rule) and policy64_q (tight bound); pi / logp against float64 on the
    kernel's own mu and the injected eps"""
    out = {k: (t.cpu().numpy() if t is not None else None)
           for k, t in eng.policy_act(obs, eps=eps, precision=fmt).items()}
    want = policy64(actor, v, vc, obs, eps)
    wq = policy64_q(actor, v, vc, obs, fmt) if fmt != "fp32" else want
    sig = dict(mu=1.0, v=float(_sig64(v.var_out)[0]), vc=float(_sig64(vc.var_out)[0]))
    msg = "%s %s:" % (label, fmt)
    errs = {}
    for k in ("mu", "v", "vc"):
        errs[k] = (_units(out[k], want[k], sig[k]), _units(out[k], wq[k], sig[k]))
        msg += " %s %.3f / %.3f" % (k, errs[k][0], errs[k][1])
    print(msg + " units (float64 / 16-bit ref)")
    for k, (e64, eq) in errs.items():
        assert e64 <= SCALE.get(fmt, 1.0), msg
        if fmt != "fp32":
            assert eq <= Q_BOUND_POLICY[fmt], msg
    ls = np.asarray(actor.log_std, F64)
    mu = out["mu"].astype(F64)
    pi = mu + eps.astype(F64) * np.exp(ls)
    assert np.allclose(out["pi"], pi, rtol=1e-5, atol=1e-6), label
    # atol: logp sums terms of O(1) and may itself be near zero
    assert np.allclose(out["logp"], _logp64(pi, mu, ls), rtol=1e-5, atol=1e-5), label
    return out


POLICY_CASES = [
    ("merged_default", {}),
    ("merged_w256", dict(a_hidden=(256, 256), hidden=(256, 256))),
    ("merged_tanh_values", dict(v_act="tanh")),
    ("merged_vc_own_scaler", dict(vc_scaler="own", v_act="tanh", vc_act="swish")),
    ("merged_vc_no_scaler", dict(vc_scaler=None)),
    ("standalone_grouped_values", dict(nv=4, nvc=4, vc_scaler="own")),       # 1 + 4 + 4 members > CMBPO_MAX_E
    ("actor64_alone", dict(a_hidden=(64, 64))),
    ("vc_relu_fp32", dict(vc_act="ReLU")),                                    # VC the tensor cores do not take
]


@pytest.mark.parametrize("name,kw", POLICY_CASES, ids=[c[0] for c in POLICY_CASES])
def test_policy_pass_vs_float64(eng, name, kw):
    actor, v, vc, obs, eps = _policy_problem(zlib.crc32(name.encode()), **kw)
    _load_policy(eng, actor, v, vc)
    for fmt in ("fp32", "fp16", "bf16"):
        _check_policy(eng, actor, v, vc, obs, eps, fmt, name)


# ---------------------------------------------------------------------------------------------------- coherence
def test_set_scalers_reaches_the_policy_pass(eng):
    """Engine.set_scalers on V and on VC changes what the fp16 / bf16 policy pass computes (the merged pack folds
    every member's input scaler into its first layer)."""
    from cmbpo_b200 import _lib as L
    actor, v, vc, obs, eps = _policy_problem(71, vc_scaler="own")
    _load_policy(eng, actor, v, vc)
    _check_policy(eng, actor, v, vc, obs, eps, "fp16", "before set_scalers")
    rng = np.random.default_rng(72)
    for which, n in ((L.NET_V, v), (L.NET_VC, vc)):
        mu = (n.mu_in.reshape(-1) + 0.3 * _sig64(n.var_in) * rng.standard_normal(n.in_dim)).astype(F32)
        var = (n.var_in.reshape(-1) * np.exp(rng.uniform(-0.7, 0.7, n.in_dim))).astype(F32)
        eng.set_scalers(which, mu, var)
        n.mu_in, n.var_in = mu.reshape(1, -1), var.reshape(1, -1)
    for fmt in ("fp32", "fp16", "bf16"):
        _check_policy(eng, actor, v, vc, obs, eps, fmt, "after set_scalers")


def test_value_training_reaches_the_policy_pass(eng):
    """B200PE.train on V (MSE, input scaler refit): afterwards the fp16 value head follows the fp32 one."""
    actor, v, vc, obs, eps = _policy_problem(73)
    policy = _load_policy(eng, actor, v, vc)
    before = eng.policy_act(obs, eps=eps, precision="fp32")["v"].cpu().numpy()
    rng = np.random.default_rng(74)
    X = (obs[rng.integers(0, obs.shape[0], 4096)] * F32(1.5)).astype(F32)
    Y = np.tanh(X[:, :3].sum(axis=1, keepdims=True)).astype(F32)
    policy.v.configure_training(loss="MSE", lr=1e-3, use_scaler_in=True)
    policy.v.train(X, Y, batch_size=256, max_epochs=3, holdout_ratio=0.1, hide_progress=True,
                   rng=np.random.RandomState(75))
    ref = eng.policy_act(obs, eps=eps, precision="fp32")["v"].cpu().numpy()
    assert not np.allclose(ref, before, rtol=1e-3, atol=1e-3)
    sig = float(_sig64(v.var_out)[0])
    for fmt in ("fp16", "bf16"):
        got = eng.policy_act(obs, eps=eps, precision=fmt)["v"].cpu().numpy()
        e = _units(got, ref, sig)
        print("trained V %s: %.3f units against fp32" % (fmt, e))
        assert e <= SCALE[fmt], (fmt, e)


def test_load_actor_reaches_the_policy_pass(eng):
    actor, v, vc, obs, eps = _policy_problem(76)
    policy = _load_policy(eng, actor, v, vc)
    _check_policy(eng, actor, v, vc, obs, eps, "fp16", "first actor")
    actor2 = _policy_problem(77)[0]
    policy.load_actor(actor2.W, actor2.b, actor2.log_std)
    for fmt in ("fp16", "bf16"):
        _check_policy(eng, actor2, v, vc, obs, eps, fmt, "second actor")


# ---------------------------------------------------------------------------------------------------- loud failures
@pytest.mark.parametrize("K0,hidden,act,D", [(20, (128, 128), "ReLU", 5), (65, (128, 128), "swish", 5),
                                             (20, (200, 256), "swish", 5), (20, (512, 512), "tanh", 64)],
                         ids=["relu", "k0_65", "mixed_widths", "out128_w512"])
def test_unsupported_dynamics_name_fp32(eng, K0, hidden, act, D):
    """out128_w512: above width 256 the tensor-memory layout holds at most 96 output columns (the OUT accumulator
    would overlap the last hidden layer's buffer; such a net used to return NaN)."""
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    ens, rng = _ensemble(80, K0, hidden, D, True, act, 3)
    model = cb.B200PE.from_arrays(eng, L.NET_DYN, ens)
    x = _rows(rng, ens, 50)
    for fmt in ("fp16", "bf16"):
        with pytest.raises(cb.CmbpoError, match="fp32"):
            model.predict_ensemble_device(x, precision=fmt)
            eng.synchronize()
    m, v = (t.cpu().numpy() for t in model.predict_ensemble_device(x, precision="fp32"))
    wm, wv = forward64(ens, x)
    assert _units(m, wm, _sig64(ens.var_out)) <= 1.0 and _vrel(v, wv) <= 1e-3


def test_3d_input_is_an_error_on_tensor_cores(eng):
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    ens, rng = _ensemble(81, 20, (128, 128), 5, True, "swish", 3)
    cb.B200PE.from_arrays(eng, L.NET_DYN, ens)
    x3 = np.stack([_rows(rng, ens, 40) for _ in range(3)])
    for fmt in ("fp16", "bf16"):
        with pytest.raises(cb.CmbpoError, match="2-D inputs only"):
            eng.predict_ensemble(L.NET_DYN, x3, precision=fmt)


def test_zero_rows_are_a_no_op(eng):
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    ens, _ = _ensemble(82, 20, (256, 256), 5, True, "swish", 3)
    cb.B200PE.from_arrays(eng, L.NET_DYN, ens)
    actor, v, vc, obs, eps = _policy_problem(83)
    _load_policy(eng, actor, v, vc)
    for fmt in ("fp32", "fp16", "bf16"):
        m, var = eng.predict_ensemble(L.NET_DYN, np.zeros((0, 20), F32), precision=fmt)
        assert m.shape == (3, 0, 5) and var.shape == (3, 0, 5)
        m, var = eng.predict_mean(L.NET_DYN, np.zeros((0, 20), F32), precision=fmt)
        assert m.shape == (0, 5)
        out = eng.policy_act(obs[:0], eps=eps[:0], precision=fmt)
        assert out["mu"].shape == (0, 6) and out["v"].shape == (0,)
        eng.synchronize()
