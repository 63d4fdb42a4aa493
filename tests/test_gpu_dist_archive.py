"""GPU, one device: sharded start-state sampling.  `DeviceArchive.sample_start_states(shard=(lo, hi))` returns
rows lo:hi of the unsharded call bit for bit, and `cmbpo_archive_sample_boltz_range` writes the entries a
whole-batch `cmbpo_archive_sample_boltz` writes at those positions, at and across the kernel's 256-sample
block boundaries."""
import numpy as np
import pytest

from oracle import cmbpo_oracle as orc

pytestmark = pytest.mark.gpu
O, A = 17, 6


def make_archive(engine, ep, seed):
    import cmbpo_b200 as cb
    rng = np.random.default_rng(seed)
    n = len(ep)
    obs = rng.standard_normal((n, O)).astype(np.float32)
    mu = (0.3 * rng.standard_normal((n, A))).astype(np.float32)
    ls = (np.linspace(-0.9, -0.2, A) + 0.05 * ep[:, None]).astype(np.float32)
    arch = cb.DeviceArchive(engine, n, O, A, seed=5)
    arch.append(obs, mu, ls, ep)
    return arch


def _policy(engine):
    import cmbpo_b200 as cb
    dyn, actor, v, vc = orc.make_problem(31, O, A, hidden=(64, 64))
    pol = cb.B200Policy(engine)
    pol.load_actor(actor.W, actor.b, actor.log_std)
    pol.load_values(v, vc)
    return pol


def test_sharded_start_states_are_rows_of_the_whole_batch(engine):
    import cmbpo_b200 as cb
    pol = _policy(engine)
    ep = np.repeat(np.arange(5, dtype=np.int32), 700)
    arch = make_archive(engine, ep, 11)
    # 512 samples: the per-epoch KL sums of two blocks, whose float64 atomics commute, so reruns give the same KLs
    B = 512
    arch._draw = 0
    full = arch.sample_start_states(pol, B, alpha=2.0)
    for shard in ((0, B), (0, 256), (256, 512), (0, 0), (512, 512), (100, 100), (1, 300), (255, 257), (3, 511)):
        arch._draw = 0
        part = arch.sample_start_states(pol, B, alpha=2.0, shard=shard)
        lo, hi = shard
        assert arch._draw == 2                       # the draw counter advances as for the whole batch
        np.testing.assert_array_equal(part["kls"], full["kls"])
        for k in ("indices", "observations", "mu", "log_std"):
            got, want = part[k].cpu().numpy(), full[k].cpu().numpy()[lo:hi]
            assert got.shape == want.shape and got.dtype == want.dtype, (k, shard)
            np.testing.assert_array_equal(got, want, err_msg="%s %s" % (k, shard))
    # a partition of the batch concatenates back to it
    parts = []
    for lo, hi in ((0, 130), (130, 130), (130, 400), (400, 512)):
        arch._draw = 0
        parts.append(arch.sample_start_states(pol, B, alpha=2.0, shard=(lo, hi))["observations"].cpu().numpy())
    np.testing.assert_array_equal(np.concatenate(parts), full["observations"].cpu().numpy())
    with pytest.raises(cb.CmbpoError):
        arch.sample_start_states(pol, B, shard=(10, B + 1))


def test_boltz_range_entry_point(engine):
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    e, t = engine, engine.torch
    ep = np.repeat(np.arange(7, dtype=np.int32), 333)
    arch = make_archive(engine, ep, 12)
    sorted_idx, offs, _ = arch._build_index()
    eps = arch.epochs_list
    cdf = np.cumsum(np.linspace(1.0, 2.0, len(eps)))
    cdf /= cdf[-1]
    eps_d, cdf_d = e.to_device(eps.astype(np.int32), t.int32), e.to_device(cdf, t.float64)
    B, seed, draw = 1300, 5, 9
    whole = e.zeros(B, dtype=t.int32)
    L.check(e.lib.cmbpo_archive_sample_boltz(e.h, e._p(sorted_idx), e._p(offs), e._p(eps_d), e._p(cdf_d), len(eps),
                                             B, seed, draw, e._p(whole)))
    whole = whole.cpu().numpy()
    assert (whole >= 0).all()
    for first, count in ((0, 256), (256, 256), (255, 1), (255, 2), (250, 300), (511, 513), (1024, 276), (0, 1300),
                         (1299, 1), (700, 0)):
        out = e.zeros(count + 1, dtype=t.int32) - 7          # one guard entry past the range
        L.check(e.lib.cmbpo_archive_sample_boltz_range(e.h, e._p(sorted_idx), e._p(offs), e._p(eps_d), e._p(cdf_d),
                                                       len(eps), first, count, seed, draw, e._p(out)))
        got = out.cpu().numpy()
        np.testing.assert_array_equal(got[:count], whole[first:first + count], err_msg=str((first, count)))
        assert got[count] == -7
    # samples past the batch one GPU would draw are the next samples of the same stream
    out = e.zeros(10, dtype=t.int32)
    L.check(e.lib.cmbpo_archive_sample_boltz_range(e.h, e._p(sorted_idx), e._p(offs), e._p(eps_d), e._p(cdf_d),
                                                   len(eps), B - 5, 10, seed, draw, e._p(out)))
    np.testing.assert_array_equal(out.cpu().numpy()[:5], whole[-5:])
    with pytest.raises(cb.CmbpoError):
        L.check(e.lib.cmbpo_archive_sample_boltz_range(e.h, e._p(sorted_idx), e._p(offs), e._p(eps_d), e._p(cdf_d),
                                                       len(eps), -1, 4, seed, draw, e._p(out)))
