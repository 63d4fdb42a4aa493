"""GPU parity of K3/K4 (GAE scans, statistics, normalisation, compaction) against the oracle.
Bar: STRICT scan bit-exact (float64 sequential = scipy lfilter order); WARP scan <= 1 float32 ulp;
statistics within float32 summation-order tolerance (stated per assert)."""
import numpy as np
import pytest

from oracle import cmbpo_oracle as orc

pytestmark = pytest.mark.gpu
G = dict(gamma=0.99, lam=0.95, cgamma=0.97, clam=0.5)


def _paths(seed, B, T, full=False):
    rng = np.random.default_rng(seed)
    rew = rng.standard_normal((B, T)).astype(np.float32)
    val = rng.standard_normal((B, T)).astype(np.float32)
    cost = (rng.random((B, T)) < 0.1).astype(np.float32)
    cval = rng.standard_normal((B, T)).astype(np.float32)
    length = np.full(B, T - 1, np.int32) if full else rng.integers(0, T, B).astype(np.int32)
    lv = rng.standard_normal(B).astype(np.float32)
    lc = rng.standard_normal(B).astype(np.float32)
    return rew, val, cost, cval, length, lv, lc


def _oracle_paths(rew, val, cost, cval, length, lv, lc):
    B, T = rew.shape
    out = [np.zeros((B, T), np.float32) for _ in range(4)]
    for L in np.unique(length):
        if L == 0:
            continue
        m = length == L
        res = orc.gae_path(rew[m, :L], val[m, :L], cost[m, :L], cval[m, :L], lv[m], lc[m],
                           G["gamma"], G["lam"], G["cgamma"], G["clam"])
        for o, r in zip(out, res):
            o[m, :L] = r
    return out


@pytest.mark.parametrize("B,T", [(1, 2), (37, 35), (4096, 35), (1000, 36), (513, 9)])
def test_gae_rows_strict_bit_exact(engine, B, T):
    import torch
    rew, val, cost, cval, length, lv, lc = _paths(B * 7 + T, B, T)
    want = _oracle_paths(rew, val, cost, cval, length, lv, lc)
    d = lambda a: engine.to_device(a)
    # reference layout [B, T] (row-major)
    got = engine.gae_paths(d(rew), d(val), d(cost), d(cval), engine.to_device(length, torch.int32),
                           d(lv), d(lc), G["gamma"], G["lam"], G["cgamma"], G["clam"], B, T, T, 1)
    for g, w in zip(got, want):
        assert np.array_equal(g.cpu().numpy(), w)
    # time-major layout [T, B] (the rollout buffers)
    tm = lambda a: engine.to_device(np.ascontiguousarray(a.T))
    got = engine.gae_paths(tm(rew), tm(val), tm(cost), tm(cval), engine.to_device(length, torch.int32),
                           d(lv), d(lc), G["gamma"], G["lam"], G["cgamma"], G["clam"], B, T, 1, B)
    for g, w in zip(got, want):
        assert np.array_equal(g.cpu().numpy().T, w)


@pytest.mark.parametrize("scan", [0, 1])
def test_gae_flat_segments(engine, scan):
    import torch
    rng = np.random.default_rng(11)
    lens = np.concatenate([rng.integers(1, 1001, 40), [0, 1, 32, 33, 64, 1000]])
    offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    n = int(offs[-1])
    rew, val, cval = (rng.standard_normal(n).astype(np.float32) for _ in range(3))
    cost = (rng.random(n) < 0.1).astype(np.float32)
    lv, lc = (rng.standard_normal(len(lens)).astype(np.float32) for _ in range(2))
    want = orc.cpobuffer_gae_flat(rew, val, cost, cval, offs, lv, lc, G["gamma"], G["lam"],
                                  G["cgamma"], G["clam"])
    d = lambda a: engine.to_device(a)
    got = engine.gae_flat(d(rew), d(val), d(cost), d(cval), engine.to_device(offs, torch.int64),
                          d(lv), d(lc), G["gamma"], G["lam"], G["cgamma"], G["clam"], scan=scan)
    for g, w in zip(got, want):
        g = g.cpu().numpy()
        if scan == 0:
            assert np.array_equal(g, w)
        else:
            assert np.all(np.abs(g - w) <= 2 * np.spacing(np.abs(w)))


def test_stats_normalise_compact(engine):
    import torch
    B, T, O = 777, 35, 17
    rng = np.random.default_rng(3)
    length = rng.integers(0, T, B).astype(np.int32)
    length[:5] = 0
    mask = np.arange(T)[None] < length[:, None]
    adv, cadv, ret, cret = (rng.standard_normal((B, T)).astype(np.float32) * 3 + 1 for _ in range(4))
    obs = rng.standard_normal((B, T, O)).astype(np.float32)
    tm = lambda a: engine.to_device(np.ascontiguousarray(np.swapaxes(a, 0, 1)))
    d_adv, d_cadv, d_ret, d_cret, d_obs = tm(adv), tm(cadv), tm(ret), tm(cret), tm(obs)
    d_len = engine.to_device(length, torch.int32)
    sums = engine.adv_statistics_device(d_adv, d_cadv, d_ret, d_cret, B, T, 1, B, d_len)
    st = engine.stats_from_sums(sums.cpu().numpy())
    mean, std = orc.stats_scalar(adv[mask])
    cmean, _ = orc.stats_scalar(cadv[mask])
    assert st["n"] == mask.sum()
    # float32 pairwise (numpy) vs float64-accumulated (device) sums: a few ulp of the mean
    assert abs(st["adv_mean"] - mean) <= 4e-7 * max(1, abs(mean))
    assert abs(st["adv_std"] - std) <= 4e-7 * std
    assert abs(st["cadv_mean"] - cmean) <= 4e-7 * max(1, abs(cmean))
    assert abs(st["ret_mean"] - ret[mask].mean()) <= 1e-6
    engine.adv_normalise_device(d_adv, d_cadv, B, T, 1, B, d_len, sums)
    want_adv = (adv - st["adv_mean"]) / (st["adv_std"] + np.float32(1e-8))
    got = d_adv.cpu().numpy().T
    assert np.array_equal(got[mask], want_adv.astype(np.float32)[mask])      # same mean/std -> bit exact
    assert np.array_equal(got[~mask], adv[~mask])                            # unpopulated untouched
    assert np.array_equal(d_cadv.cpu().numpy().T[mask], (cadv - st["cadv_mean"])[mask])
    off = engine.path_offsets(d_len)
    assert np.array_equal(off.cpu().numpy(), np.concatenate([[0], np.cumsum(length)]))
    n_rows = int(off[-1])
    flat = engine.compact(d_obs, B, T, O, d_len, off, n_rows).cpu().numpy()
    assert np.array_equal(flat, obs[mask])                                   # numpy boolean-mask order
    flat1 = engine.compact(d_ret, B, T, 1, d_len, off, n_rows).cpu().numpy()
    assert np.array_equal(flat1, ret[mask])


def test_statistics_of_empty_batch_touch_nothing(engine):
    """adv_statistics_device / adv_normalise_device on a batch without valid entries: n == 0, nothing is touched."""
    import torch
    B, T = 913, 35
    rng = np.random.default_rng(5)
    adv, cadv, ret, cret = (rng.standard_normal((B, T)).astype(np.float32) * 2 - 0.3 for _ in range(4))
    tm = lambda a: engine.to_device(np.ascontiguousarray(np.swapaxes(a, 0, 1)))
    zero = engine.to_device(np.zeros(B, np.int32), torch.int32)
    a, c = tm(adv), tm(cadv)
    sums = engine.adv_statistics_device(a, c, tm(ret), tm(cret), B, T, 1, B, zero)
    engine.adv_normalise_device(a, c, B, T, 1, B, zero, sums)
    assert engine.stats_from_sums(sums.cpu().numpy())["n"] == 0
    assert np.array_equal(a.cpu().numpy().T, adv) and np.array_equal(c.cpu().numpy().T, cadv)


def test_path_offsets_large(engine):
    import torch
    rng = np.random.default_rng(1)
    length = rng.integers(0, 35, 300001).astype(np.int32)
    off = engine.path_offsets(engine.to_device(length, torch.int32)).cpu().numpy()
    assert np.array_equal(off, np.concatenate([[0], np.cumsum(length.astype(np.int64))]))
