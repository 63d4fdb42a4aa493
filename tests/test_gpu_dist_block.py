"""-m gpu: the model-rollout block of algorithms/cmbpo.py:241-270 (archive sample -> reset -> sample(max_samples)
loop with the caller's stop rule -> finish_all_paths -> get) sharded over G ranks with ModelSampler.distribute()
gives the one-GPU result, gathered on rank 0.

Transports: NCCL with one GPU per rank (2 ranks, and 4 when 4 GPUs are visible; skipped otherwise, like
test_gpu_nccl2.py), and gloo with every rank on GPU 0 (2 and 4 ranks: the same library code, the messages go
through host memory), so that one GPU runs the multi-rank logic too.

Against one GPU on the same seeded archive and weights, for HCS and AntSafe (terminations), uncertainty and
schedule mode, max_samples none / a cut inside rank 0's shard / a cut that straddles ranks, fp16 and fp32:
root rows bit for bit (adv / cadv: the tolerance of test_gpu_nccl2.py, their statistics are all-reduced),
zero-row arrays elsewhere, sample() calls, sample counts and alive ratios exact, diagnostics counts and maxima
exact and float64 sums within rtol 1e-12, compute_dynamics_dkl identical on every rank and within rtol 1e-12
of one GPU.  The uncertainty limit both runs use is the one-GPU value, so a last-bit difference of the
calibration cannot move a threshold."""
import os
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

B, T, N_ARCH, STOP = 1200, 8, 3000, 0.1
GAE = dict(gamma=0.99, lam=0.95, cost_gamma=0.97, cost_lam=0.5)
TASKS = {"hcs": ("HalfCheetahSafe-v2", 17, 6), "ant": ("AntSafe-v2", 29, 8)}
PRECISIONS = ("fp16", "fp32")
MODES = ("uncertainty", "schedule")
CAPS = (None, "inside", "straddle")
CASES = [(k, m, c, p) for k in TASKS for m in MODES for c in CAPS for p in PRECISIONS]
TRANSPORTS = [("gloo", 2), ("gloo", 4), ("nccl", 2), ("nccl", 4)]
EXACT_DIAG = ("pool-size", "msampler/samples_added", "msampler/rollout_H_max", "msampler/max_path_return",
              "msampler/max_dkl", "msampler/rollout_H_mean")


class _ShapeEnv:
    class _S:
        def __init__(self, n):
            self.shape = (n,)

    def __init__(self, O, A):
        self.observation_space, self.action_space = self._S(O), self._S(A)


def _setup(dev, key, precision):
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L, workload as wl
    task, O, A = TASKS[key]
    dyn, actor, v, vc = wl.make_problem(21, O, A, hidden=(512, 512), task=task)
    eng = cb.Engine(dev, precision=precision)
    model = cb.B200PE.from_arrays(eng, L.NET_DYN, dyn)
    policy = cb.B200Policy(eng)
    policy.load_actor(actor.W, actor.b, actor.log_std)
    policy.load_values(v, vc)
    obs, _ = wl.make_states(22, N_ARCH, O, A, dyn)
    rng = np.random.default_rng(23)
    mu = (0.3 * rng.standard_normal((N_ARCH, A))).astype(np.float32)
    ls = np.broadcast_to(actor.log_std, (N_ARCH, A)) + 0.1 * rng.standard_normal((N_ARCH, A))
    ep = np.repeat(np.arange(4, dtype=np.int32), N_ARCH // 4)
    return dict(eng=eng, model=model, policy=policy, task=task, O=O, A=A,
                archive=(obs, mu, ls.astype(np.float32), ep))


def _block(s, mode, lim, max_samples, shard, distributed):
    """One rollout block; `lim` None: the uncertainty limit is 4 x this run's calibrated dkl."""
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L
    eng, O, A = s["eng"], s["O"], s["A"]
    arch = cb.DeviceArchive(eng, N_ARCH, O, A, seed=9)
    arch.append(*s["archive"])
    env = cb.FakeEnv(_ShapeEnv(O, A), s["task"], s["model"], True, True, False)
    pool = cb.ModelBuffer(shard[1] - shard[0], O, A, T, engine=eng)
    pool.initialize({"mu": (A,), "log_std": (A,)}, **GAE)
    smp = cb.ModelSampler(T, B, mode, seed=3)
    smp.initialize(env, s["policy"], pool)
    if distributed:
        smp.distribute()
    start = arch.sample_start_states(s["policy"], B, alpha=1.0, shard=shard)["observations"]
    dkl = smp.compute_dynamics_dkl(start)
    lim = 4.0 * dkl if lim is None else lim
    smp.set_rollout_dkl(lim)
    smp.reset(start)
    calls, ratios = 0, []
    while True:                                           # algorithms/cmbpo.py:258-263
        _, _, _, info = smp.sample(max_samples)
        calls += 1
        ratios.append(info["alive_ratio"])
        if max_samples and smp._total_samples >= 0.99 * max_samples:
            break
        if info["alive_ratio"] <= STOP:
            break
    diag = dict(smp.finish_all_paths())
    capped = int((pool.bufs.end_reason == L.END_CAPPED).sum().item())
    lengths = pool.bufs.length.cpu().numpy()
    out, bdiag = pool.get()
    return dict(out=out, bdiag=bdiag, diag=diag, dkl=dkl, lim=lim, calls=calls, ratios=ratios,
                total=smp._total_samples, capped=capped, lengths=lengths)


def _cap(lengths, cap, world):
    """max_samples whose cut at step 1 takes a part of rank 0's survivors (inside) or all of them and a part of
    rank 1's (straddle), from the path lengths of the run without a cap (survivors of step t: length > t)."""
    from cmbpo_b200.dist import shard_bounds
    if cap is None:
        return None
    s = [int((lengths[slice(*shard_bounds(B, r, world))] > 1).sum()) for r in (0, 1)]
    assert min(s) >= 2, s
    n = s[0] // 2 if cap == "inside" else s[0] + s[1] // 2
    return int((lengths > 0).sum() + (lengths > 1).sum() - n)


def _free_port():
    sk = socket.socket()
    sk.bind(("127.0.0.1", 0))
    port = sk.getsockname()[1]
    sk.close()
    return port


def _worker(rank, world, backend, port, jobs, q):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    import torch
    import torch.distributed as dist
    dev = rank if backend == "nccl" else 0
    torch.cuda.set_device(dev)
    kw = dict(device_id=torch.device("cuda", dev)) if backend == "nccl" else {}
    dist.init_process_group(backend, rank=rank, world_size=world, **kw)
    from cmbpo_b200.dist import shard_bounds
    shard = shard_bounds(B, rank, world)
    setups = {}
    for case, lim, max_samples in jobs:
        key, mode, _, prec = case
        if (key, prec) not in setups:
            setups[(key, prec)] = _setup(dev, key, prec)
        r = _block(setups[(key, prec)], mode, lim, max_samples, shard, True)
        if rank != 0:
            r["out"] = [(a.shape, a.dtype) for a in r["out"]]
        q.put((case, rank, r))
    dist.barrier()
    dist.destroy_process_group()
    for s in setups.values():
        s["eng"].close()


_RESULTS = {}


def _results(backend, world):
    """{case: (one-GPU result, [rank results])}, computed once per transport."""
    import torch
    if (backend, world) in _RESULTS:
        return _RESULTS[(backend, world)]
    if backend == "nccl" and torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    import torch.multiprocessing as mp
    refs, jobs, setups = {}, [], {}
    for case in CASES:
        key, mode, cap, prec = case
        if (key, prec) not in setups:
            setups[(key, prec)] = _setup(0, key, prec)
        s = setups[(key, prec)]
        if ("free", key, mode, prec) not in _RESULTS:          # the one-GPU run without a cap
            _RESULTS[("free", key, mode, prec)] = _block(s, mode, None, None, (0, B), False)
        free = _RESULTS[("free", key, mode, prec)]
        ms = _cap(free["lengths"], cap, world)
        refs[case] = free if cap is None else _block(s, mode, free["lim"], ms, (0, B), False)
        jobs.append((case, free["lim"], ms))
    for s in setups.values():
        s["eng"].close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, backend, port, jobs, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = {}
    for _ in range(world * len(jobs)):
        case, rank, r = q.get(timeout=600)
        got.setdefault(case, [None] * world)[rank] = r
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    _RESULTS[(backend, world)] = {c: (refs[c], got[c]) for c in CASES}
    return _RESULTS[(backend, world)]


@pytest.mark.parametrize("backend,world", TRANSPORTS)
@pytest.mark.parametrize("key,mode,cap,precision", CASES)
def test_sharded_block_equals_one_gpu(backend, world, key, mode, cap, precision):
    ref, ranks = _results(backend, world)[(key, mode, cap, precision)]
    # the case covers what it names: the cap cuts inside rank 0's shard, or on rank 0 and rank 1
    if cap is not None:
        assert ref["capped"] > 0 and ranks[0]["capped"] > 0
        assert (ranks[1]["capped"] > 0) == (cap == "straddle")
        assert sum(r["capped"] for r in ranks) == ref["capped"]
    assert 1 < ref["calls"] < T
    root = ranks[0]
    for i, (g, w) in enumerate(zip(root["out"], ref["out"])):
        assert g.shape == w.shape and g.dtype == w.dtype, i
        if i in (2, 3):                                   # adv, cadv
            np.testing.assert_allclose(g, w, rtol=2e-6, atol=2e-6, err_msg=str(i))
        else:
            np.testing.assert_array_equal(g, w, err_msg=str(i))
    for r in ranks[1:]:
        for (shape, dtype), w in zip(r["out"], ref["out"]):
            assert shape == (0,) + w.shape[1:] and dtype == w.dtype
    for r in ranks:
        assert r["calls"] == ref["calls"] and r["total"] == ref["total"]
        assert r["ratios"] == ref["ratios"]
        assert r["dkl"] == root["dkl"]
        np.testing.assert_allclose(r["dkl"], ref["dkl"], rtol=1e-12)
        assert r["diag"] == root["diag"] and r["bdiag"] == root["bdiag"]
        assert r["bdiag"]["poolm_batch_size"] == ref["bdiag"]["poolm_batch_size"] == len(ref["out"][0])
        for k in ("poolm_ret_mean", "poolm_cret_mean"):
            np.testing.assert_allclose(r["bdiag"][k], ref["bdiag"][k], rtol=3e-7, atol=1e-9)
        assert r["diag"].keys() == ref["diag"].keys()
        for k, w in ref["diag"].items():
            if k in EXACT_DIAG:
                assert r["diag"][k] == w, k
            else:
                np.testing.assert_allclose(r["diag"][k], w, rtol=1e-12, atol=1e-300, err_msg=k)
