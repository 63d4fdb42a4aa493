"""-m gpu: checkpoint and resume.  A run saved with checkpoint.save_state, loaded into a new Engine and continued gives
the bits of the same run without the break:

  * ensemble training (B200PE.train with the scalers re-fitted, so that the running merge crosses the save): the
    weights, Adam moments, step count, elites and val_loss after a second train() call, for the HCS dynamics
    ensemble 7 x (512, 512) MSPE and V 3 x (128, 128) MSE, in fp32, TF32 and bf16 and fp32 -> save -> bf16 (the bf16
    weight copy is rebuilt from the restored master weights); one case saves in another Python process;
  * the rollout block (DeviceArchive.sample_start_states, ModelSampler.reset / sample / finish_all_paths,
    ModelBuffer.get) of the batch after the save, at fp16 and fp32, on one GPU and sharded over two gloo ranks that
    each load rank 0's file and call distribute().
Also: cmbpo_ens_train_state_set / _get, the bf16 weight copy rebuilt after _set, the rejections, and a trained
B200PE written with write_pe_checkpoint and read back with load_pe predicting bit for bit."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import cmbpo_oracle as orc

pytestmark = pytest.mark.gpu

TESTS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(TESTS)

# name: (E, hidden, probabilistic)
NETS = {"hcs": (7, (512, 512), True), "v": (3, (128, 128), False)}
MATHS = ("fp32", "tf32", "bf16", "fp32>bf16")
N_ROWS, EPOCHS, BS = 2048, 2, 256


def _net(engine, name):
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    E, hidden, prob = NETS[name]
    if prob:
        dyn, _, _, _ = orc.make_problem(31, 17, 6, hidden=hidden, num_nets=E, num_elites=5, gain=1.0)
        return cb.B200PE.from_arrays(engine, L.NET_DYN, dyn), L.NET_DYN, 23, 18
    _, _, v, _ = orc.make_problem(31, 17, 6, hidden=(64, 64), vf_nets=E, vf_hidden=hidden, gain=1.0)
    return cb.B200PE.from_arrays(engine, L.NET_V, v, name="VEnsemble"), L.NET_V, 17, 1


def _data(din, dout):
    rng = np.random.default_rng(5)
    X = (rng.standard_normal((N_ROWS, din)) * 2.0 + 0.5).astype(np.float32)
    M = (rng.standard_normal((din, dout)) * 0.3).astype(np.float32)
    return X, (np.tanh(X @ M) + 0.05 * rng.standard_normal((N_ROWS, dout))).astype(np.float32)


def _configure(model, math):
    model.configure_training(lr=1e-3, decay=1e-4, use_scaler_in=True, use_scaler_out=True, math=math)


def _train(model, rng, X, Y):
    return model.train(X, Y, batch_size=BS, max_epochs=EPOCHS, holdout_ratio=0.1, rng=rng)


def _maths(math):
    return math.split(">") if ">" in math else (math, math)


def _first_half(name, math):
    """A new run's first train() call; returns (the state to save, engine)."""
    import cmbpo_b200 as cb
    eng = cb.Engine(0, precision="fp32")
    model, which, din, dout = _net(eng, name)
    _configure(model, _maths(math)[0])
    rng = np.random.RandomState(17)
    _train(model, rng, *_data(din, dout))
    n, keys, pos, g, c = rng.get_state()
    return {"pe": model.state_dict(), "rng": {"name": n, "keys": keys, "pos": pos, "has_gauss": g,
                                              "cached_gaussian": c}}, eng


def _second_half(model, rng, math):
    """The second train() call; fp32>bf16 switches to bf16 first."""
    first, second = _maths(math)
    if second != first:
        _configure(model, second)
    out = _train(model, rng, *_data(model.in_dim, model._d))
    return _result(model, out)


def _result(model, out):
    sd = model.state_dict()
    return dict(layers=sd["layers"], step=sd["step"], elites=list(model.elite_inds),
                val_loss=out["%s/val_loss" % model.name], cache=sd["train"]["scaler_cache"])


def _uninterrupted(name, math):
    import cmbpo_b200 as cb
    eng = cb.Engine(0, precision="fp32")
    model, which, din, dout = _net(eng, name)
    _configure(model, _maths(math)[0])
    rng = np.random.RandomState(17)
    _train(model, rng, *_data(din, dout))
    r = _second_half(model, rng, math)
    eng.close()
    return r


def _resume(path, name):
    import cmbpo_b200 as cb
    sd = cb.load_state(path)
    eng = cb.Engine(0, precision="fp32")
    from cmbpo_b200 import _lib as L
    model = cb.B200PE.from_state_dict(eng, L.NET_DYN if NETS[name][2] else L.NET_V, sd["pe"])
    r = sd["rng"]
    rng = np.random.RandomState()
    rng.set_state((r["name"], r["keys"], r["pos"], r["has_gauss"], r["cached_gaussian"]))
    return model, rng, eng


def _assert_same(a, b):
    assert a["step"] == b["step"] > 0
    assert a["elites"] == b["elites"]
    assert a["val_loss"] == b["val_loss"]
    for l, (x, y) in enumerate(zip(a["layers"], b["layers"])):
        assert sorted(x) == sorted(y) == ["W", "b", "mW", "mb", "vW", "vb"]
        for k in x:
            assert x[k].dtype == np.float32 and np.array_equal(x[k], y[k]), (l, k)
    for k in ("in", "out"):
        x, y = a["cache"][k], b["cache"][k]
        assert x["count"] == y["count"] > 0
        assert np.array_equal(x["mean"], y["mean"]) and np.array_equal(x["var"], y["var"])


@pytest.mark.parametrize("math", MATHS)
@pytest.mark.parametrize("name", list(NETS))
def test_training_continues_bit_identically(tmp_path, name, math):
    import cmbpo_b200 as cb
    state, eng = _first_half(name, math)
    path = str(tmp_path / "run.npz")
    cb.save_state(path, state)
    eng.close()
    model, rng, eng2 = _resume(path, name)
    got = _second_half(model, rng, math)
    eng2.close()
    _assert_same(got, _uninterrupted(name, math))


def _child_save(path, name, math):
    """Run in a separate process: the first half, saved."""
    import cmbpo_b200 as cb
    state, eng = _first_half(name, math)
    cb.save_state(path, state)
    eng.close()


def test_training_resumes_in_another_process(tmp_path):
    name, math = "hcs", "bf16"
    path = str(tmp_path / "run.npz")
    code = ("import sys; sys.path[:0] = [%r, %r]; import test_gpu_resume as m; m._child_save(%r, %r, %r)"
            % (ROOT, TESTS, path, name, math))
    subprocess.run([sys.executable, "-c", code], check=True, cwd=ROOT, timeout=600)
    model, rng, eng = _resume(path, name)
    got = _second_half(model, rng, math)
    eng.close()
    _assert_same(got, _uninterrupted(name, math))


# ---- the C entry points ---------------------------------------------------------------------------------------------
def test_train_state_set_get_and_bf16_repack():
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    eng = cb.Engine(0, precision="fp32")
    model, which, din, dout = _net(eng, "hcs")
    nl = len(eng.nets[which]["dims"]) - 1
    assert eng.train_state_get(which, 0) == (None, -1)
    rng = np.random.default_rng(2)
    mom = []
    for l in range(nl):
        K, H = eng.nets[which]["dims"][l:l + 2]
        E = eng.nets[which]["E"]
        mom.append([rng.standard_normal(s).astype(np.float32) for s in ((E, K, H), (E, K, H), (E, H), (E, H))])
        mom[-1][1], mom[-1][3] = np.abs(mom[-1][1]), np.abs(mom[-1][3])
        eng.train_state_set(which, l, *mom[-1], 41)
    for l in range(nl):
        got, step = eng.train_state_get(which, l)
        assert step == 41
        for g, w in zip(got, mom[l]):
            assert np.array_equal(g.cpu().numpy(), w)
    # the first bf16 step after _set rebuilds the bf16 weight copy (L more launches), the next does not
    X, Y = _data(din, dout)
    x = eng.to_device(np.ascontiguousarray(np.broadcast_to(X[:BS], (7, BS, din))))
    y = eng.to_device(np.ascontiguousarray(np.broadcast_to(Y[:BS], (7, BS, dout))))
    _configure(model, "bf16")

    def launches():
        n0 = eng.launch_count
        eng.train_step(which, x, y, model._train_cfg)
        return eng.launch_count - n0

    assert launches() == 4 * nl + 2
    assert launches() == 3 * nl + 2
    assert eng.train_state_get(which, 0)[1] == 43
    eng.train_state_set(which, 0, *mom[0], 3)            # on an existing state
    assert launches() == 4 * nl + 2
    assert launches() == 3 * nl + 2
    assert eng.train_state_get(which, 1)[1] == 5
    # rejections: bad slot, bad layer, negative step, a slot that is not loaded
    lib, h = eng.lib, eng.h
    assert lib.cmbpo_ens_train_state_set(h, 9, 0, None, None, None, None, 0) != 0
    assert lib.cmbpo_ens_train_state_set(h, which, nl, None, None, None, None, 0) != 0
    assert lib.cmbpo_ens_train_state_set(h, which, -1, None, None, None, None, 0) != 0
    assert lib.cmbpo_ens_train_state_set(h, which, 0, None, None, None, None, -1) != 0
    assert b"step" in lib.cmbpo_last_error()
    assert lib.cmbpo_ens_train_state_set(h, L.NET_VC, 0, None, None, None, None, 0) != 0
    assert b"not loaded" in lib.cmbpo_last_error()
    with pytest.raises(ValueError):
        eng.train_state_set(which, 0, mom[1][0], *mom[0][1:], 1)
    eng.close()


def test_precision_mismatch_is_refused(tmp_path):
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    eng = cb.Engine(0, precision="fp16")
    model, which, _, _ = _net(eng, "v")
    sd = model.state_dict()
    assert sd["precision"] == "fp16" and sd["step"] == -1 and sd["train"] is None
    eng.close()
    other = cb.Engine(0, precision="fp32")
    with pytest.raises(ValueError, match="precision"):
        cb.B200PE.from_state_dict(other, L.NET_V, sd)
    other.close()


# ---- the rollout block ------------------------------------------------------------------------------------------
B, T, N_ARCH, STOP = 1200, 8, 3000, 0.1
GAE = dict(gamma=0.99, lam=0.95, cost_gamma=0.97, cost_lam=0.5)
TASK, O, A = "HalfCheetahSafe-v2", 17, 6


class _ShapeEnv:
    class _S:
        def __init__(self, n):
            self.shape = (n,)

    def __init__(self, O, A):
        self.observation_space, self.action_space = self._S(O), self._S(A)


def _world(precision):
    """Engine, models, policy, archive and sampler of a new run."""
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L, workload as wl
    dyn, actor, v, vc = wl.make_problem(21, O, A, hidden=(512, 512), task=TASK)
    eng = cb.Engine(0, precision=precision)
    model = cb.B200PE.from_arrays(eng, L.NET_DYN, dyn)
    policy = cb.B200Policy(eng, seed=4)
    policy.load_actor(actor.W, actor.b, actor.log_std)
    policy.load_values(v, vc)
    obs, _ = wl.make_states(22, N_ARCH, O, A, dyn)
    rng = np.random.default_rng(23)
    mu = (0.3 * rng.standard_normal((N_ARCH, A))).astype(np.float32)
    ls = (np.broadcast_to(actor.log_std, (N_ARCH, A)) + 0.1 * rng.standard_normal((N_ARCH, A))).astype(np.float32)
    arch = cb.DeviceArchive(eng, N_ARCH + 500, O, A, seed=9)
    arch.append(obs[:2000], mu[:2000], ls[:2000], np.repeat(np.arange(2, dtype=np.int32), 1000))
    arch.append(obs[2000:], mu[2000:], ls[2000:], np.repeat(np.arange(2, 4, dtype=np.int32), 500))
    smp = cb.ModelSampler(T, B, "uncertainty", seed=3)
    return dict(eng=eng, model=model, policy=policy, arch=arch, smp=smp)


def _attach(w, shard=(0, B), distributed=False):
    import cmbpo_b200 as cb
    env = cb.FakeEnv(_ShapeEnv(O, A), TASK, w["model"], True, True, False)
    pool = cb.ModelBuffer(shard[1] - shard[0], O, A, T, engine=w["eng"])
    pool.initialize({"mu": (A,), "log_std": (A,)}, **GAE)
    w["smp"].initialize(env, w["policy"], pool)
    if distributed:
        w["smp"].distribute()
    return w


def _block(w, shard=(0, B)):
    smp, pool = w["smp"], w["smp"].pool
    start = w["arch"].sample_start_states(w["policy"], B, alpha=1.0, shard=shard)["observations"]
    dkl = smp.compute_dynamics_dkl(start)
    smp.set_rollout_dkl(4.0 * dkl)
    smp.reset(start)
    infos = []
    while True:                                           # algorithms/cmbpo.py:258-263
        _, _, _, info = smp.sample()
        infos.append(info)
        if info["alive_ratio"] <= STOP:
            break
    diag = dict(smp.finish_all_paths())
    out, bdiag = pool.get()
    return dict(out=out, bdiag=bdiag, diag=diag, dkl=dkl, infos=infos)


def _save_world(w):
    return {"dyn": w["model"].state_dict(), "v": w["policy"].v.state_dict(), "vc": w["policy"].vc.state_dict(),
            "policy": w["policy"].state_dict(), "archive": w["arch"].state_dict(), "sampler": w["smp"].state_dict()}


def _load_world(sd, precision):
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    eng = cb.Engine(0, precision=precision)
    model = cb.B200PE.from_state_dict(eng, L.NET_DYN, sd["dyn"])
    v = cb.B200PE.from_state_dict(eng, L.NET_V, sd["v"])
    vc = cb.B200PE.from_state_dict(eng, L.NET_VC, sd["vc"])
    policy = cb.B200Policy.from_state_dict(eng, sd["policy"], v, vc)
    arch = cb.DeviceArchive.from_state_dict(eng, sd["archive"])
    return dict(eng=eng, model=model, policy=policy, arch=arch, smp=cb.ModelSampler.from_state_dict(sd["sampler"]))


_ROLLOUT = {}


def _rollout_runs(precision, tmp_dir):
    """(second block of the uninterrupted run, its state file after the first block)."""
    if precision not in _ROLLOUT:
        import cmbpo_b200 as cb
        w = _attach(_world(precision))
        _block(w)
        path = os.path.join(tmp_dir, "rollout_%s.npz" % precision)
        cb.save_state(path, _save_world(w))
        second = _block(w)
        # the sampler refuses a state taken while a batch is in flight
        w["smp"].reset(w["arch"].sample_start_states(w["policy"], B)["observations"])
        with pytest.raises(cb.CmbpoError, match="in flight"):
            w["smp"].state_dict()
        w["eng"].close()
        _ROLLOUT[precision] = (second, path)
    return _ROLLOUT[precision]


def _assert_block_equal(got, want, adv_tol=None):
    for i, (g, x) in enumerate(zip(got["out"], want["out"])):
        assert g.shape == x.shape and g.dtype == x.dtype, i
        if adv_tol and i in (2, 3):                       # adv, cadv: the statistics are all-reduced
            np.testing.assert_allclose(g, x, rtol=adv_tol, atol=adv_tol, err_msg=str(i))
        else:
            assert np.array_equal(g, x), i
    assert got["dkl"] == want["dkl"]
    assert [i["alive_ratio"] for i in got["infos"]] == [i["alive_ratio"] for i in want["infos"]]
    assert [i["ensemble_dkl_mean"] for i in got["infos"]] == [i["ensemble_dkl_mean"] for i in want["infos"]]


@pytest.mark.parametrize("precision", ["fp16", "fp32"])
def test_rollout_after_restore_is_bit_identical(tmp_path_factory, precision):
    import cmbpo_b200 as cb
    want, path = _rollout_runs(precision, str(tmp_path_factory.mktemp("rollout")))
    w = _attach(_load_world(cb.load_state(path), precision))
    got = _block(w)
    w["eng"].close()
    assert 1 < len(want["infos"]) < T
    _assert_block_equal(got, want)
    assert got["bdiag"] == want["bdiag"]
    assert got["diag"].keys() == want["diag"].keys()
    for k in want["diag"]:
        assert got["diag"][k] == want["diag"][k], k


def _free_port():
    import socket
    sk = socket.socket()
    sk.bind(("127.0.0.1", 0))
    port = sk.getsockname()[1]
    sk.close()
    return port


def _worker(rank, world, port, path, precision, q):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    import torch
    import torch.distributed as dist
    import cmbpo_b200 as cb
    from cmbpo_b200.dist import shard_bounds
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    shard = shard_bounds(B, rank, world)
    w = _attach(_load_world(cb.load_state(path), precision), shard, distributed=True)
    r = _block(w, shard)
    if rank != 0:
        r["out"] = [(a.shape, a.dtype) for a in r["out"]]
    q.put((rank, r))
    dist.barrier()
    dist.destroy_process_group()
    w["eng"].close()


def test_sharded_rollout_after_restore_equals_one_gpu(tmp_path_factory):
    import torch.multiprocessing as mp
    precision, world = "fp16", 2
    want, path = _rollout_runs(precision, str(tmp_path_factory.mktemp("rollout")))
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, path, precision, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=600) for _ in range(world))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    _assert_block_equal(got[0], want, adv_tol=2e-6)
    for (shape, dtype), x in zip(got[1]["out"], want["out"]):
        assert shape == (0,) + x.shape[1:] and dtype == x.dtype
    for r in got.values():
        assert r["dkl"] == got[0]["dkl"] and r["diag"] == got[0]["diag"]
        assert r["diag"]["msampler/samples_added"] == want["diag"]["msampler/samples_added"]


# ---- export to the reference's format ---------------------------------------------------------------------------
def test_written_pe_checkpoint_predicts_bit_identically(tmp_path):
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    eng = cb.Engine(0, precision="fp32")
    model, which, din, dout = _net(eng, "hcs")
    _configure(model, "bf16")
    X, Y = _data(din, dout)
    _train(model, np.random.RandomState(1), X, Y)
    cb.write_pe_checkpoint(str(tmp_path), "BNN", 3, model)
    eng2 = cb.Engine(0, precision="fp32")
    back = cb.load_pe(eng2, L.NET_DYN, str(tmp_path), "BNN", 3, elite_inds=model.elite_inds)
    for prec in ("fp32", "fp16"):
        for a, b in zip(model.predict_ensemble_device(X[:700], precision=prec),
                        back.predict_ensemble_device(X[:700], precision=prec)):
            assert np.array_equal(a.cpu().numpy(), b.cpu().numpy()), prec
        for a, b in zip(model.predict_device(X[:700], precision=prec), back.predict_device(X[:700], precision=prec)):
            assert np.array_equal(a.cpu().numpy(), b.cpu().numpy()), prec
    eng.close()
    eng2.close()
