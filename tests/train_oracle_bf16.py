"""TEST INFRASTRUCTURE (oracle): the bf16 training step of csrc/train_tc.cu restated in float64.

The step of oracle/train_oracle.py with `round_bf16=True` rounding to bf16 exactly where the kernels round: the
scaled input, the weight copy the GEMMs read, the hidden activations, and each gradient with respect to a
pre-activation where it becomes a GEMM operand.  Everything else stays float64 (the kernels keep it fp32): bias
addition, pre-activations, raw outputs, loss, the bias gradients (sums of the unrounded gradient), dW, Adam.
With `round_bf16=False` every function here gives the bits of its oracle/train_oracle.py counterpart
(tests/test_train_oracle_bf16_cpu.py checks that).  It lives beside the tests rather than as a keyword of
oracle/train_oracle.py so that the pinned reference oracle stays byte for byte as it is; it reuses that module's
activations, loss parts and Adam, and restates only forward / grads / train_step with the rounding points.
"""
import numpy as np

from oracle import train_oracle as tro


def bf16(x):
    """Round to bf16 (round-to-nearest-even from the float32 value, as the kernels' conversions), as float64."""
    f = np.ascontiguousarray(x, dtype=np.float32)
    u = f.view(np.uint32).astype(np.uint64)
    r = (((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16).astype(np.uint32).view(np.float32)
    return np.where(np.isnan(f), f, r).astype(np.float64)


def _rounding(round_bf16):
    return bf16 if round_bf16 else (lambda a: a)


def forward(W, b, acts, x, mu_in=None, var_in=None, round_bf16=False):
    """tro.forward; hs[l] is the (rounded) operand the layer-l GEMMs read."""
    rnd = _rounding(round_bf16)
    a = rnd(x if mu_in is None else (x - mu_in) / tro.sigma(var_in))
    zs, hs = [], [a]
    for l, (Wl, bl, act) in enumerate(zip(W, b, acts)):
        z = np.einsum("ebi,eio->ebo", a, rnd(Wl)) + bl.reshape(Wl.shape[0], 1, -1)
        zs.append(z)
        a = tro.ACT[act][0](z)
        if l + 1 < len(W):                     # the raw outputs the loss reads stay unrounded
            a = rnd(a)
        hs.append(a)
    return zs, hs


def grads(W, b, acts, x, y, loss, mu_in=None, var_in=None, mu_out=None, var_out=None, round_bf16=False):
    """tro.grads: loss vector [E] and the gradients of sum_e loss_e (decays excluded) for every W_l, b_l."""
    rnd = _rounding(round_bf16)
    zs, hs = forward(W, b, acts, x, mu_in, var_in, round_bf16)
    out = zs[-1]
    yt = y if mu_out is None else (y - mu_out) / tro.sigma(var_out)
    E, bs = out.shape[0], out.shape[1]
    D = yt.shape[-1]
    n = bs * D
    if loss == "MSPE":
        mean, logvar, s, v, q, ratio = tro.mspe_parts(out, yt)
        lvec = tro.mspe_loss_vector(out, yt)
        g = np.concatenate([2.0 * (mean - yt) / n, (2.0 * ratio * (v - s) * v + 0.1 * logvar) / n], axis=-1)
    else:
        lvec = tro.mse_loss_vector(out, yt)
        g = (out - yt) / n
    gW, gb = [None] * len(W), [None] * len(W)
    for l in range(len(W) - 1, -1, -1):
        gb[l] = g.sum(axis=1)
        g = rnd(g)
        gW[l] = np.einsum("ebi,ebo->eio", hs[l], g)
        if l > 0:
            g = np.einsum("ebo,eio->ebi", g, rnd(W[l])) * tro.ACT[acts[l - 1]][1](zs[l - 1])
    return lvec, gW, gb


def train_step(W, b, acts, x, y, loss, opt, decay, round_bf16=False, **scalers):
    """tro.train_step with the gradients of `grads` above."""
    lvec, gW, gb = grads(W, b, acts, x, y, loss, round_bf16=round_bf16, **scalers)
    wd = tro.decay_coeffs(len(W), decay)
    params, gs = [], []
    for l in range(len(W)):
        params += [W[l], b[l]]
        gs += [gW[l] + wd[l] * W[l], gb[l].reshape(b[l].shape)]
    new = opt.step(params, gs)
    return lvec, new[0::2], new[1::2], gW, gb
