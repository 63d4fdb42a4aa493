"""cmbpo_rollout flags that must not change a result: alive-row compaction (bit for bit against
ROLLOUT_NO_COMPACT), the retired ROLLOUT_FUSE bit, and ROLLOUT_NO_STORE (the same per-path results and
step statistics without the per-step fields)."""
import numpy as np
import pytest

from oracle import cmbpo_oracle as orc
from helpers import TASKS, GAE, load_problem, ShapeEnv, calibrated_dkl_lim

pytestmark = pytest.mark.gpu

FIELDS = ("length", "end_reason", "last_val", "last_cval", "obs", "nextobs", "act", "mu", "rew", "val", "cval",
          "logp", "cost", "dkl", "dyn_error", "term", "adv", "ret", "cadv", "cret", "cum_dkl", "path_return",
          "path_cost", "final_obs", "step_stats")


def _run(engine, cfg, B, T, O, A, obs, flags, prec, **kw):
    import cmbpo_b200 as cb
    bufs = cb.RolloutBuffers(engine, B, T, O, A)
    bufs.set_inputs(obs)
    bufs.run(cfg, precision=prec, flags=flags, **kw)
    bufs.gae(GAE["gamma"], GAE["lam"], GAE["cost_gamma"], GAE["cost_lam"])
    engine.synchronize()
    return bufs


def _assert_identical(engine, a, b, skip=()):
    t = engine.torch
    for name in FIELDS:
        if name in skip:
            continue
        x, y = getattr(a, name), getattr(b, name)
        if name == "step_stats":        # float64 sums accumulated with atomics: the order differs
            assert t.allclose(x, y, rtol=1e-12, atol=0), name
            continue
        assert bool(t.equal(x, y)), name


@pytest.mark.parametrize("key,hidden,B", [("hcs", (512, 512), 40000), ("ant", (256, 256), 20000), ("hum", (128, 128), 3000)])
def test_flags_do_not_change_bits_philox_uncertainty(engine, key, hidden, B):
    """Philox noise, the reference's default 'uncertainty' rollout mode (paths end at many different steps),
    many tiles per CTA and tiles shared by two CTAs (B >> 148 * 128): alive-row compaction and the retired
    ROLLOUT_FUSE bit give the same bits as the run without compaction."""
    from cmbpo_b200 import _lib as L
    import cmbpo_b200 as cb
    task, O, A = TASKS[key]
    T = 20
    dyn, actor, v, vc = orc.make_problem(311, O, A, hidden=hidden, task=task)
    model, _ = load_problem(engine, dyn, actor, v, vc)
    env = cb.FakeEnv(ShapeEnv(O, A), task, model, True, True, False)
    obs, act = orc.make_states(312, B, O, A, dyn)
    lim = calibrated_dkl_lim(dyn, task, obs[:2000], act[:2000], factor=12.0)
    cfg = env.env_cfg(True)
    kw = dict(uncertainty_mode=True, dkl_lim=lim, seed=5)
    ref = _run(engine, cfg, B, T, O, A, obs, L.ROLLOUT_NO_COMPACT, "fp16", **kw)
    ln = ref.length.cpu().numpy()
    assert 1 < ln.mean() < T - 2 and len(np.unique(ln)) > 5
    for flags in (0, L.ROLLOUT_FUSE):
        got = _run(engine, cfg, B, T, O, A, obs, flags, "fp16", **kw)
        # final_obs of ended paths is whatever row the compaction left behind: compare alive paths only
        _assert_identical(engine, got, ref, skip=("final_obs",))


def test_no_store_mode_gives_the_same_statistics(engine):
    """ROLLOUT_NO_STORE: per-path results and step statistics without the per-step fields."""
    from cmbpo_b200 import _lib as L
    task, O, A = TASKS["ant"]
    B, T = 2000, 8
    dyn, actor, v, vc = orc.make_problem(331, O, A, hidden=(512, 512), task=task)
    load_problem(engine, dyn, actor, v, vc)
    obs, act = orc.make_states(332, B, O, A, dyn)
    cfg = L.EnvCfg(L.TERM_ANTSAFE, L.COST_ANTSAFE, 0, 1, 1)
    t = engine.torch
    for prec in ("fp32", "fp16"):
        full = _run(engine, cfg, B, T, O, A, obs, 0, prec, seed=3)
        lean = _run(engine, cfg, B, T, O, A, obs, L.ROLLOUT_NO_STORE, prec, seed=3)
        for name in ("length", "end_reason", "last_val", "last_cval", "cum_dkl", "path_return", "path_cost"):
            assert bool(t.equal(getattr(full, name), getattr(lean, name))), (prec, name)
        assert t.allclose(full.step_stats, lean.step_stats, rtol=1e-12, atol=0)
        assert float(lean.rew.abs().sum().item()) == 0.0 and float(lean.nextobs.abs().sum().item()) == 0.0
