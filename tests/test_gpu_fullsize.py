"""GPU, at BASELINE.json's full sizes, where the oracle cannot run the whole workload in seconds:
size-independent properties of the rollout / GAE path, plus oracle checks on random subsets.

  * trajectory chaining: obs[t+1] == next_obs[t] bit-exactly, lengths / end reasons consistent
  * determinism and shard invariance: the same (seed, global path id) gives the same bits whether a
    path is computed in one 100 k batch or in a shard with `path_id_base`
  * the H-step entry point agrees with the single-step entry points on step 0
  * GAE of the device rollout equals the oracle's float64 scan bit-exactly on sampled paths
  * advantage normalisation: mean 0 / std 1 (mpi_statistics_scalar semantics), compaction order
  * the standalone GAE workloads of SURVEY.md section 8d config 4 (ModelBuffer [32768, 35] with ragged
    lengths, CPOBuffer flat 1049 x 1000) bit-exact against the oracle
"""
import numpy as np
import pytest

from oracle import cmbpo_oracle as orc
from helpers import TASKS, GAE, load_problem, calibrated_dkl_lim

pytestmark = pytest.mark.gpu
F32 = np.float32


@pytest.fixture(scope="module")
def hcs_full(engine):
    """HCS, 100 000 start states, maxroll 35, (512,512) ensemble, fp16 tensor-core path."""
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    task, O, A = TASKS["hcs"]
    B, T = 100000, 35
    dyn, actor, v, vc = orc.make_problem(0, O, A, hidden=(512, 512), task=task)
    model, policy = load_problem(engine, dyn, actor, v, vc)
    obs, _ = orc.make_states(1, B, O, A, dyn)
    cfg = L.EnvCfg(L.TERM_NO_DONE, L.COST_HCS, 0, 1, 1)
    bufs = cb.RolloutBuffers(engine, B, T, O, A)
    bufs.set_inputs(obs)
    bufs.run(cfg, seed=99, precision="fp16")
    bufs.gae(GAE["gamma"], GAE["lam"], GAE["cost_gamma"], GAE["cost_lam"])
    engine.synchronize()
    return dict(bufs=bufs, cfg=cfg, obs=obs, dyn=dyn, actor=actor, v=v, vc=vc, B=B, T=T, O=O, A=A,
                model=model, policy=policy)


def test_fullsize_chain_and_lengths(hcs_full, engine):
    from cmbpo_b200 import _lib as L
    b, B, T = hcs_full["bufs"], hcs_full["B"], hcs_full["T"]
    ln = b.length.cpu().numpy()
    assert (ln == T - 1).all()                                   # no_done + dkl_lim = inf: horizon only
    assert (b.end_reason.cpu().numpy() == L.END_HORIZON).all()
    t = engine.torch
    assert bool(t.equal(b.obs[1:T - 1], b.nextobs[0:T - 2]))    # s_{t+1} of step t is s_t of step t+1
    assert bool(t.equal(b.obs[0], engine.to_device(hcs_full["obs"], t.float32)))
    assert bool(t.isfinite(b.nextobs[:T - 1]).all()) and bool(t.isfinite(b.adv[:T - 1]).all())
    assert float(b.obs[T - 1].abs().max()) == 0.0                # column maxroll-1 is never populated
    cost = b.cost[:T - 1]
    assert bool(((cost == 0) | (cost == 1)).all())               # hcs_cost_f is an indicator
    want = (t.abs(b.nextobs[:T - 1, :, -1] * 10.0) < 2.0).to(t.float32)
    assert bool(t.equal(cost, want))                             # statics.py:10-15 on the stored next_obs


def test_fullsize_determinism_and_shard_invariance(hcs_full, engine):
    import cmbpo_b200 as cb
    b, B, T, O, A = (hcs_full[k] for k in ("bufs", "B", "T", "O", "A"))
    t = engine.torch
    lo, hi = 37000, 37000 + 4096
    shard = cb.RolloutBuffers(engine, hi - lo, T, O, A)
    shard.set_inputs(hcs_full["obs"][lo:hi])
    shard.run(hcs_full["cfg"], seed=99, path_id_base=lo, precision="fp16")
    shard.gae(GAE["gamma"], GAE["lam"], GAE["cost_gamma"], GAE["cost_lam"])
    engine.synchronize()
    # the tensor-core kernel tiles 128 rows: rows land in different tiles / lanes in the shard, and an
    # MMA row's result does not depend on its tile neighbours -> bit-identical
    for name in ("obs", "nextobs", "act", "mu", "rew", "val", "cval", "logp", "cost", "dkl", "adv", "cadv"):
        full = getattr(b, name)[:, lo:hi]
        assert bool(t.equal(full, getattr(shard, name))), name
    again = cb.RolloutBuffers(engine, hi - lo, T, O, A)
    again.set_inputs(hcs_full["obs"][lo:hi])
    again.run(hcs_full["cfg"], seed=99, path_id_base=lo, precision="fp16")
    engine.synchronize()
    assert bool(t.equal(again.nextobs, shard.nextobs)) and bool(t.equal(again.logp, shard.logp))
    other = cb.RolloutBuffers(engine, hi - lo, T, O, A)
    other.set_inputs(hcs_full["obs"][lo:hi])
    other.run(hcs_full["cfg"], seed=100, path_id_base=lo, precision="fp16")
    engine.synchronize()
    assert not bool(t.equal(other.act, shard.act))               # a different seed draws different noise


def test_fullsize_step0_matches_single_step_entry_points(hcs_full, engine):
    """cmbpo_rollout's first step == cmbpo_fakeenv_step on (obs, the action the rollout took)."""
    b, cfg = hcs_full["bufs"], hcs_full["cfg"]
    t = engine.torch
    rows = np.random.default_rng(3).choice(hcs_full["B"], 8192, replace=False)
    r = engine.to_device(rows.astype(np.int64), t.int64)
    obs0, act0 = b.obs[0][r].contiguous(), b.act[0][r].contiguous()
    out = engine.fakeenv_step(cfg, obs0, act0, path_ids=engine.to_device(rows.astype(np.int32), t.int32),
                              seed=99, step=0, precision="fp16")
    assert bool(t.equal(out["next_obs"], b.nextobs[0][r]))
    assert bool(t.equal(out["rew"], b.rew[0][r])) and bool(t.equal(out["cost"], b.cost[0][r]))
    assert bool(t.equal(out["dkl_path"], b.dkl[0][r]))
    # and against the oracle on a subset (fp16 operands: the single-step tolerance of test_gpu_tc.py)
    sub = rows[:1024]
    dyn = hcs_full["dyn"]
    x = np.concatenate([b.obs[0].cpu().numpy()[sub], b.act[0].cpu().numpy()[sub]], -1)
    wm, wv = orc.pe_forward(dyn, x)
    sig = np.maximum(np.sqrt(dyn.var_out), 1e-2)
    gm = hcs_full["model"].predict_ensemble_device(engine.to_device(x, t.float32), precision="fp16")[0].cpu().numpy()
    assert np.all(np.abs(gm - wm) <= 1e-3 * np.abs(wm) + 1e-3 * sig)


def test_fullsize_gae_bit_exact_on_sampled_paths(hcs_full):
    b, T = hcs_full["bufs"], hcs_full["T"]
    rows = np.random.default_rng(4).choice(hcs_full["B"], 512, replace=False)
    f = {k: getattr(b, k).cpu().numpy()[:T - 1, rows].T.copy() for k in ("rew", "val", "cost", "cval", "adv", "ret", "cadv", "cret")}
    lv, lc = b.last_val.cpu().numpy()[rows], b.last_cval.cpu().numpy()[rows]
    adv, ret, cadv, cret = orc.gae_path(f["rew"], f["val"], f["cost"], f["cval"], lv, lc,
                                        GAE["gamma"], GAE["lam"], GAE["cost_gamma"], GAE["cost_lam"])
    for name, want in (("adv", adv), ("ret", ret), ("cadv", cadv), ("cret", cret)):
        assert np.array_equal(f[name], want), name


def test_fullsize_normalise_and_compaction(hcs_full, engine):
    b, B, T, O = (hcs_full[k] for k in ("bufs", "B", "T", "O"))
    t = engine.torch
    adv, cadv = b.adv.clone(), b.cadv.clone()
    sums = engine.adv_statistics_device(adv, cadv, b.ret, b.cret, B, T, 1, B, b.length)
    st = engine.stats_from_sums(sums.cpu().numpy())
    assert st["n"] == B * (T - 1)
    ref_mean = float(b.adv[:T - 1].double().mean())
    assert abs(st["adv_mean"] - ref_mean) <= 1e-6 * max(1.0, abs(ref_mean)) + 1e-6
    engine.adv_normalise_device(adv, cadv, B, T, 1, B, b.length, sums)
    a = adv[:T - 1].double()
    assert abs(float(a.mean())) < 1e-4 and abs(float(a.std(unbiased=False)) - 1.0) < 1e-3
    assert abs(float(cadv[:T - 1].double().mean())) < 1e-4
    off = engine.path_offsets(b.length)
    n_rows = int(off[-1].item())
    assert n_rows == B * (T - 1)
    flat = engine.compact(b.obs, B, T, O, b.length, off, n_rows)
    # ModelBuffer.get(): buf[populated_mask] is path-major, then time (modelbuffer.py:218)
    for p in (0, 1, 12345, B - 1):
        assert bool(t.equal(flat[p * (T - 1):(p + 1) * (T - 1)], b.obs[:T - 1, p]))


def test_fullsize_ant_uncertainty_histogram(engine):
    """AntSafe (terminations + uncertainty cut-off), 125 000 start states = one rank's share of the
    1 M-state config: path lengths, end reasons and the populated mask stay consistent."""
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    task, O, A = TASKS["ant"]
    B, T = 125000, 35
    dyn, actor, v, vc = orc.make_problem(2, O, A, hidden=(512, 512), task=task)
    load_problem(engine, dyn, actor, v, vc)
    obs, act = orc.make_states(3, B, O, A, dyn)
    lim = calibrated_dkl_lim(dyn, task, obs[:2000], act[:2000], factor=12.0)
    cfg = L.EnvCfg(L.TERM_ANTSAFE, L.COST_ANTSAFE, 0, 1, 1)
    bufs = cb.RolloutBuffers(engine, B, T, O, A)
    bufs.set_inputs(obs)
    bufs.run(cfg, uncertainty_mode=True, dkl_lim=lim, seed=5, precision="fp16")
    bufs.gae(GAE["gamma"], GAE["lam"], GAE["cost_gamma"], GAE["cost_lam"])
    engine.synchronize()
    t = engine.torch
    ln, er = bufs.length.cpu().numpy(), bufs.end_reason.cpu().numpy()
    h_len, h_unc = bufs.histogram()
    assert np.array_equal(h_len, np.bincount(ln, minlength=T + 1))
    assert np.array_equal(h_unc, np.bincount(ln[er == L.END_UNCERTAIN], minlength=T + 1))
    assert set(np.unique(er)) <= {L.END_UNCERTAIN, L.END_HORIZON, L.END_TERMINAL}
    assert (ln[er == L.END_HORIZON] == T - 1).all() and (ln[er != L.END_HORIZON] <= T - 1).all()
    assert len(np.unique(ln)) > 3                                 # the workload really is ragged
    term = bufs.term.cpu().numpy().astype(bool)                   # [T, B]
    idx = np.nonzero(er == L.END_TERMINAL)[0]
    assert term[ln[idx] - 1, idx].all()                           # a terminal path ends on its done step
    pop = np.arange(T)[:, None] < ln[None, :]
    assert not term[pop & ~(np.arange(T)[:, None] == (ln - 1)[None, :])].any()   # and nowhere before
    cum = bufs.cum_dkl.cpu().numpy()
    assert (cum[er != L.END_UNCERTAIN] < lim).all()               # stored steps stay below the limit
    lv = bufs.last_val.cpu().numpy()
    assert (lv[er == L.END_TERMINAL] == 0).all()                  # model_sampler.py:364: reward bootstrap 0
    # unpopulated cells are zero (modelbuffer.py:53-98)
    assert float(bufs.rew.cpu().numpy()[~pop].__abs__().max(initial=0.0)) == 0.0
    # GAE bit-exact on sampled ragged paths
    rows = np.random.default_rng(6).choice(B, 256, replace=False)
    for p in rows:
        n = ln[p]
        if n == 0:
            continue
        f = {k: getattr(bufs, k)[:n, p].cpu().numpy() for k in ("rew", "val", "cost", "cval", "adv", "cret")}
        adv, ret, cadv, cret = orc.gae_path(f["rew"], f["val"], f["cost"], f["cval"],
                                            F32(bufs.last_val[p].item()), F32(bufs.last_cval[p].item()),
                                            GAE["gamma"], GAE["lam"], GAE["cost_gamma"], GAE["cost_lam"])
        assert np.array_equal(f["adv"], adv) and np.array_equal(f["cret"], cret)
    del t


def test_standalone_gae_config4(engine):
    """SURVEY.md section 8d config 4: 1 048 576 steps as ModelBuffer [32768, 35] rows with ragged
    lengths (row-major, the reference's layout), and as a CPOBuffer flat buffer of 1049 x 1000."""
    t = engine.torch
    rng = np.random.default_rng(7)
    B, T = 32768, 35
    rew, val, cval = (rng.standard_normal((B, T)).astype(F32) for _ in range(3))
    cost = (rng.random((B, T)) < 0.1).astype(F32)
    ln = rng.integers(1, T, B).astype(np.int32)
    ln[:64] = T - 1
    lv, lc = rng.standard_normal(B).astype(F32), rng.standard_normal(B).astype(F32)
    d = {k: engine.to_device(x, t.float32) for k, x in dict(rew=rew, val=val, cost=cost, cval=cval, lv=lv, lc=lc).items()}
    out = engine.gae_paths(d["rew"], d["val"], d["cost"], d["cval"], engine.to_device(ln, t.int32), d["lv"], d["lc"],
                           GAE["gamma"], GAE["lam"], GAE["cost_gamma"], GAE["cost_lam"], B, T,
                           path_stride=T, time_stride=1)
    got = [x.cpu().numpy() for x in out]
    for p in rng.choice(B, 2048, replace=False):
        n = ln[p]
        want = orc.gae_path(rew[p, :n], val[p, :n], cost[p, :n], cval[p, :n], lv[p], lc[p],
                            GAE["gamma"], GAE["lam"], GAE["cost_gamma"], GAE["cost_lam"])
        for g, w in zip(got, want):
            assert np.array_equal(g[p, :n], w)
    # CPOBuffer: 1049 paths x 1000 steps, strict scan bit-exact, warp scan within 1 ulp
    from cmbpo_b200 import _lib as L
    n_seg, seg = 1049, 1000
    n = n_seg * seg
    r2, v2, cv2 = (rng.standard_normal(n).astype(F32) for _ in range(3))
    c2 = (rng.random(n) < 0.1).astype(F32)
    off = np.arange(n_seg + 1, dtype=np.int64) * seg
    lv2, lc2 = rng.standard_normal(n_seg).astype(F32), rng.standard_normal(n_seg).astype(F32)
    dd = [engine.to_device(x, t.float32) for x in (r2, v2, c2, cv2)]
    strict = engine.gae_flat(*dd, engine.to_device(off, t.int64), engine.to_device(lv2, t.float32),
                             engine.to_device(lc2, t.float32), GAE["gamma"], GAE["lam"], GAE["cost_gamma"],
                             GAE["cost_lam"], scan=L.SCAN_STRICT)
    warp = engine.gae_flat(*dd, engine.to_device(off, t.int64), engine.to_device(lv2, t.float32),
                           engine.to_device(lc2, t.float32), GAE["gamma"], GAE["lam"], GAE["cost_gamma"],
                           GAE["cost_lam"], scan=L.SCAN_WARP)
    pick = rng.choice(n_seg, 48, replace=False)
    sub_off = np.concatenate([[0], np.cumsum(np.full(len(pick), seg))])
    sel = np.concatenate([np.arange(off[i], off[i + 1]) for i in pick])
    want = orc.cpobuffer_gae_flat(r2[sel], v2[sel], c2[sel], cv2[sel], sub_off, lv2[pick], lc2[pick],
                                  GAE["gamma"], GAE["lam"], GAE["cost_gamma"], GAE["cost_lam"])
    for g, gw, w in zip(strict, warp, want):
        g, gw = g.cpu().numpy()[sel], gw.cpu().numpy()[sel]
        assert np.array_equal(g, w)
        assert np.all(np.abs(gw - w) <= np.spacing(np.abs(w)) + 1e-30)


def test_alive_row_compaction_is_invisible(engine):
    """Squeezing finished paths out of the batch (tensor-core path, AntSafe + uncertainty cut-off) must
    not change a single bit: a row's result does not depend on which tile / lane it occupies."""
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    task, O, A = TASKS["ant"]
    B, T = 20000, 35
    dyn, actor, v, vc = orc.make_problem(12, O, A, hidden=(512, 512), task=task)
    load_problem(engine, dyn, actor, v, vc)
    obs, act = orc.make_states(13, B, O, A, dyn)
    lim = calibrated_dkl_lim(dyn, task, obs[:2000], act[:2000], factor=30.0)
    cfg = L.EnvCfg(L.TERM_ANTSAFE, L.COST_ANTSAFE, 0, 1, 1)
    t = engine.torch
    res = []
    for flags in (0, L.ROLLOUT_NO_COMPACT):
        bufs = cb.RolloutBuffers(engine, B, T, O, A)
        bufs.set_inputs(obs)
        bufs.run(cfg, uncertainty_mode=True, dkl_lim=lim, seed=21, precision="fp16", flags=flags)
        bufs.gae(GAE["gamma"], GAE["lam"], GAE["cost_gamma"], GAE["cost_lam"])
        engine.synchronize()
        res.append(bufs)
    a, b = res
    ln = a.length.cpu().numpy()
    assert 4 < ln.mean() < T - 3 and len(np.unique(ln)) > 8       # paths really end at many different steps
    for name in ("length", "end_reason", "last_val", "last_cval", "obs", "nextobs", "act", "mu", "rew", "val", "cval",
                 "logp", "cost", "dkl", "dyn_error", "term", "adv", "ret", "cadv", "cret", "cum_dkl"):
        assert bool(t.equal(getattr(a, name), getattr(b, name))), name
