"""CPU: pins the bf16 training-step oracle (tests/train_oracle_bf16.py).  Its rounding equals torch's float -> bf16
conversion (round-to-nearest-even) on random values, ties, subnormals, infinities and NaN; with rounding off it
gives the bits of oracle/train_oracle.py; with rounding on, every GEMM operand it uses is a bf16 value."""
import numpy as np
import pytest
import torch

from oracle import train_oracle as tro
import train_oracle_bf16 as trb


def _torch_bf16(x):
    return torch.tensor(x).to(torch.bfloat16).to(torch.float64).numpy()


def _same(a, b):
    np.testing.assert_array_equal(np.isnan(a), np.isnan(b))
    ok = ~np.isnan(a)
    assert np.array_equal(a[ok], b[ok])
    assert np.array_equal(np.signbit(a[ok]), np.signbit(b[ok]))


def test_bf16_rounding_matches_torch():
    rng = np.random.default_rng(0)
    base = rng.standard_normal(20000).astype(np.float32) * np.float32(10.0) ** rng.integers(-30, 30, 20000).astype(np.float32)
    # ties: bf16 keeps the top 16 bits, so bit 15 set with the low 15 bits clear is exactly half an ulp
    hi = rng.integers(0, 1 << 16, 4000, dtype=np.uint64)
    ties = ((hi << 16) | 0x8000).astype(np.uint32).view(np.float32)
    ties = ties[np.isfinite(ties)]
    tiny = np.float32(np.finfo(np.float32).tiny)
    sub = np.concatenate([rng.uniform(-1, 1, 2000).astype(np.float32) * tiny,
                          np.arange(1, 2000, dtype=np.uint32).view(np.float32)])
    special = np.array([np.inf, -np.inf, np.nan, -np.nan, 0.0, -0.0, np.finfo(np.float32).max,
                        -np.finfo(np.float32).max, 3.3895e38, 1.0, -1.0], np.float32)
    for x in (base, ties, sub, special, -ties, -sub):
        _same(trb.bf16(x), _torch_bf16(x))
    x64 = rng.standard_normal(5000) * 1e3            # float64 input: rounded through float32, as torch does
    _same(trb.bf16(x64), _torch_bf16(x64))


def _problem(seed, prob, E=3, bs=9, Din=5, H=70, D=2):
    rng = np.random.default_rng(seed)
    dims = [Din, H, H, 2 * D if prob else D]
    W = [rng.standard_normal((E, dims[i], dims[i + 1])) * 0.3 for i in range(3)]
    b = [rng.standard_normal((E, dims[i + 1])) * 0.1 for i in range(3)]
    x = rng.standard_normal((E, bs, Din))
    y = rng.standard_normal((E, bs, D))
    sc = dict(mu_in=rng.standard_normal((1, Din)), var_in=rng.uniform(0.5, 2, (1, Din)),
              mu_out=rng.standard_normal((1, D)), var_out=rng.uniform(0.5, 2, (1, D)))
    return W, b, ["swish", "tanh", None], x, y, sc


@pytest.mark.parametrize("prob", [True, False])
def test_rounding_off_is_the_float64_oracle(prob):
    W, b, acts, x, y, sc = _problem(1, prob)
    loss = "MSPE" if prob else "MSE"
    _same_all = lambda u, v: [_same(np.asarray(p), np.asarray(q)) for p, q in zip(u, v)]
    z0, h0 = tro.forward(W, b, acts, x, sc["mu_in"], sc["var_in"])
    z1, h1 = trb.forward(W, b, acts, x, sc["mu_in"], sc["var_in"], round_bf16=False)
    _same_all(z0, z1)
    _same_all(h0, h1)
    opt0 = tro.Adam([p for l in range(3) for p in (W[l], b[l])])
    opt1 = tro.Adam([p for l in range(3) for p in (W[l], b[l])])
    Wa, ba, Wb, bb = W, b, W, b
    for _ in range(3):
        r0 = tro.train_step(Wa, ba, acts, x, y, loss, opt0, 1e-2, **sc)
        r1 = trb.train_step(Wb, bb, acts, x, y, loss, opt1, 1e-2, round_bf16=False, **sc)
        _same(r0[0], r1[0])
        for k in range(1, 5):
            _same_all(r0[k], r1[k])
        Wa, ba, Wb, bb = r0[1], r0[2], r1[1], r1[2]


def test_rounding_on_rounds_every_gemm_operand():
    W, b, acts, x, y, sc = _problem(2, True)
    zs, hs = trb.forward(W, b, acts, x, sc["mu_in"], sc["var_in"], round_bf16=True)
    for h in hs[:-1]:
        _same(h, trb.bf16(h))
    assert not np.array_equal(hs[-1], trb.bf16(hs[-1]))       # raw outputs stay unrounded
    lv0, gW0, gb0 = tro.grads(W, b, acts, x, y, "MSPE", **sc)
    lv1, gW1, gb1 = trb.grads(W, b, acts, x, y, "MSPE", round_bf16=True, **sc)
    # the rounding moves results by about bf16's relative precision, no more
    for l in range(3):
        assert 0 < np.abs(gW1[l] - gW0[l]).max() <= 0.05 * np.abs(gW0[l]).max()
        assert np.abs(gb1[l] - gb0[l]).max() <= 0.05 * np.abs(gb0[l]).max()
    np.testing.assert_allclose(lv1, lv0, rtol=0.05)
