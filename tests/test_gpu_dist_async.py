"""-m gpu: ModelBuffer.get_async() on a rollout block sharded over G ranks with ModelSampler.distribute() gives, on the
root, what one GPU's get() gives for the same batch, and zero-row arrays elsewhere.

Each case runs K consecutive blocks in a pipelined order: result() of batch i-1 comes after get_async() of batch i,
so two handles are outstanding at once, and after the reset (start states, rollout queued) of the next batch.  Once
with one sampler / buffer pair per rank, in INTEGRATION.md's loop (reset, sample loop and finish_all_paths of batch
i, get_async(), result() of batch i-1), and once with two pairs on two engines (two CUDA streams) used alternately,
as bench.py's e2e_pipelined does (the reset of batch i+1 comes before the sample loop of batch i).

Transports: gloo with every rank on GPU 0 (1, 2 and 4 ranks; one rank is distribute() on a one-process group) and
NCCL with one GPU per rank (2 and 4 ranks, skipped when fewer GPUs are visible).  The reference is one GPU running the
same pairs (same archive seeds, sampler seeds and draws) with the blocking get().

Per batch: the root's arrays equal the reference bit for bit (adv / cadv within rtol / atol 2e-6: their statistics
are all-reduced), the other ranks' arrays have zero rows and the reference's dtypes and trailing shapes, get()'s and
finish_all_paths()'s diagnostics are the same on every rank, and the arrays read through result() are still intact
just before the next get_async() that may reuse their page-locked buffers."""
import os
import queue
import socket
import time

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

B, T, N_ARCH, STOP, K = 1200, 8, 3000, 0.1, 4
GAE = dict(gamma=0.99, lam=0.95, cost_gamma=0.97, cost_lam=0.5)
TASKS = {"hcs": ("HalfCheetahSafe-v2", 17, 6), "ant": ("AntSafe-v2", 29, 8)}
MODES = ("uncertainty", "schedule")
CAPS = (None, "straddle")
CASES = ([(k, m, c, "fp16") for k in TASKS for m in MODES for c in CAPS]
         + [("hcs", m, c, "fp32") for m in MODES for c in CAPS])
PAIRS = (1, 2)
TRANSPORTS = [("gloo", 1), ("gloo", 2), ("gloo", 4), ("nccl", 2), ("nccl", 4)]


class _ShapeEnv:
    class _S:
        def __init__(self, n):
            self.shape = (n,)

    def __init__(self, O, A):
        self.observation_space, self.action_space = self._S(O), self._S(A)


def _setup(dev, key, precision, stream):
    """An engine whose kernels run on `stream`, with the dynamics model and the policy of the test problem."""
    import torch
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L, workload as wl
    task, O, A = TASKS[key]
    dyn, actor, v, vc = wl.make_problem(21, O, A, hidden=(512, 512), task=task)
    with torch.cuda.stream(stream):
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
    return dict(eng=eng, model=model, policy=policy, task=task, O=O, A=A, stream=stream,
                archive=(obs, mu, ls.astype(np.float32), ep))


def _pair(s, k, mode, lim, shard, distributed):
    """Sampler / buffer pair k (its own archive and sampler seed) on the engine of setup `s`."""
    import torch
    import cmbpo_b200 as cb
    O, A = s["O"], s["A"]
    with torch.cuda.stream(s["stream"]):
        arch = cb.DeviceArchive(s["eng"], N_ARCH, O, A, seed=9 + k)
        arch.append(*s["archive"])
        env = cb.FakeEnv(_ShapeEnv(O, A), s["task"], s["model"], True, True, False)
        pool = cb.ModelBuffer(shard[1] - shard[0], O, A, T, engine=s["eng"])
        pool.initialize({"mu": (A,), "log_std": (A,)}, **GAE)
        smp = cb.ModelSampler(T, B, mode, seed=3 + k)
        smp.initialize(env, s["policy"], pool)
        if distributed:
            smp.distribute()
        smp.set_rollout_dkl(lim)
    return dict(s=s, arch=arch, pool=pool, smp=smp, shard=shard)


def _reset(p):
    import torch
    with torch.cuda.stream(p["s"]["stream"]):
        start = p["arch"].sample_start_states(p["s"]["policy"], B, alpha=1.0, shard=p["shard"])["observations"]
        p["smp"].reset(start)


def _finish(p, max_samples):
    """The sample loop of algorithms/cmbpo.py:258-263 and finish_all_paths; (diagnostics, capped paths, lengths)."""
    import torch
    from cmbpo_b200 import _lib as L
    smp, bufs = p["smp"], p["pool"].bufs
    with torch.cuda.stream(p["s"]["stream"]):
        while True:
            _, _, _, info = smp.sample(max_samples)
            if max_samples and smp._total_samples >= 0.99 * max_samples:
                break
            if info["alive_ratio"] <= STOP:
                break
        diag = dict(smp.finish_all_paths())
        capped = int((bufs.end_reason == L.END_CAPPED).sum().item())
        return diag, capped, bufs.length.cpu().numpy()


def _sequential(setups, mode, lim, caps):
    """The reference: K blocks on one GPU with the blocking get(), batch i on pair i % len(setups)."""
    pairs = [_pair(s, k, mode, lim, (0, B), False) for k, s in enumerate(setups)]
    res = []
    for i in range(K):
        p = pairs[i % len(pairs)]
        _reset(p)
        diag, capped, lengths = _finish(p, caps[i])
        out, bdiag = p["pool"].get()
        res.append(dict(out=out, bdiag=bdiag, diag=diag, capped=capped, lengths=lengths))
    return res


def _pipelined(setups, mode, lim, caps, shard):
    """K blocks in INTEGRATION.md's pipelined order with get_async(), batch i on pair i % len(setups).  Returns the
    per-batch results (arrays copied at result()) and the wall time of the loop."""
    import torch
    pairs = [_pair(s, k, mode, lim, shard, True) for k, s in enumerate(setups)]
    res, handles, held, queued = [None] * K, [], None, 0
    t0 = time.perf_counter()
    for i in range(K):
        # one pair: batch i is reset after get_async() of batch i-1; two pairs: batch i+1 is reset (its rollout
        # queued on the other pair's stream) before batch i is sampled
        while queued < min(K, i + len(pairs)):
            _reset(pairs[queued % len(pairs)])
            queued += 1
        p = pairs[i % len(pairs)]
        diag, capped, _ = _finish(p, caps[i])
        if held is not None:
            # the last arrays read through result(): a handle and a reset were issued since, and their page-locked
            # buffers are reused at the earliest by the get_async() below
            j, views = held
            res[j]["intact"] = all(np.array_equal(v, c) for v, c in zip(views, res[j]["out"]))
        with torch.cuda.stream(p["s"]["stream"]):
            handles.append((i, diag, capped, p["pool"].get_async()))
        while len(handles) == 2 or (i == K - 1 and handles):
            j, dg, cp, h = handles.pop(0)
            out, bdiag = h.result()
            res[j] = dict(out=[a.copy() for a in out], bdiag=bdiag, diag=dg, capped=cp, intact=None)
            held = (j, out)
    seconds = time.perf_counter() - t0
    return res, seconds


def _cap(lengths, world):
    """max_samples whose cut at step 1 takes all of rank 0's survivors and a part of rank 1's, from the path lengths
    of the batch without a cap (survivors of step t: length > t).  One rank: the same cut as for two."""
    from cmbpo_b200.dist import shard_bounds
    world = max(world, 2)
    s = [int((lengths[slice(*shard_bounds(B, r, world))] > 1).sum()) for r in (0, 1)]
    assert min(s) >= 2, s
    return int((lengths > 0).sum() + (lengths > 1).sum() - (s[0] + s[1] // 2))


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
    for (case, n_pairs), lim, caps in jobs:
        key, mode, _, prec = case
        for k in range(n_pairs):
            if (key, prec, k) not in setups:
                stream = torch.cuda.current_stream(dev) if k == 0 else torch.cuda.Stream(device=dev)
                setups[(key, prec, k)] = _setup(dev, key, prec, stream)
        res, seconds = _pipelined([setups[(key, prec, k)] for k in range(n_pairs)], mode, lim, caps, shard)
        if rank != 0:
            for r in res:
                r["out"] = [(a.shape, a.dtype) for a in r["out"]]
        q.put(((case, n_pairs), rank, res, seconds))
    dist.barrier()
    dist.destroy_process_group()
    for s in setups.values():
        s["eng"].close()


_RESULTS = {}


def _results(backend, world):
    """{(case, pairs): (one-GPU results, [rank results], [rank seconds])}, computed once per transport."""
    import torch
    if (backend, world) in _RESULTS:
        return _RESULTS[(backend, world)]
    if backend == "nccl" and torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    import torch.multiprocessing as mp
    stream = torch.cuda.current_stream(0)
    setups = {}
    for key, _, _, prec in CASES:
        if (key, prec) not in setups:
            setups[(key, prec)] = _setup(0, key, prec, stream)
    refs, jobs = {}, []
    for case in CASES:
        key, mode, cap, prec = case
        s = setups[(key, prec)]
        if ("lim", key, mode, prec) not in _RESULTS:      # uncertainty limit: 4 x the one-GPU calibrated dkl
            p = _pair(s, 0, mode, 0.0, (0, B), False)
            start = p["arch"].sample_start_states(s["policy"], B, alpha=1.0)["observations"]
            _RESULTS[("lim", key, mode, prec)] = 4.0 * p["smp"].compute_dynamics_dkl(start)
        lim = _RESULTS[("lim", key, mode, prec)]
        for n_pairs in PAIRS:
            free_key = ("free", key, mode, prec, n_pairs)
            if free_key not in _RESULTS:
                _RESULTS[free_key] = _sequential([s] * n_pairs, mode, lim, [None] * K)
            free = _RESULTS[free_key]
            caps = [None] * K if cap is None else [_cap(r["lengths"], world) for r in free]
            cap_key = ("capped", key, mode, prec, n_pairs, max(world, 2))
            if cap is not None and cap_key not in _RESULTS:
                _RESULTS[cap_key] = _sequential([s] * n_pairs, mode, lim, caps)
            refs[(case, n_pairs)] = free if cap is None else _RESULTS[cap_key]
            jobs.append(((case, n_pairs), lim, caps))
    for s in setups.values():
        s["eng"].close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, backend, port, jobs, q)) for r in range(world)]
    for p in procs:
        p.start()
    got, secs = {}, {}
    try:
        for _ in range(world * len(jobs)):
            while True:
                try:
                    job, rank, r, seconds = q.get(timeout=5)
                    break
                except queue.Empty:
                    dead = [p.exitcode for p in procs if p.exitcode not in (None, 0)]
                    assert not dead, "a rank exited with %s" % dead
            got.setdefault(job, [None] * world)[rank] = r
            secs.setdefault(job, [None] * world)[rank] = seconds
    except BaseException:
        for p in procs:           # the other ranks wait in a collective for the one that failed
            p.terminate()
            p.join(timeout=30)
        raise
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for key, mode, cap, prec in CASES:
        if cap is None and prec == "fp16":
            print("get_async pipelined, %s %d ranks, %s %s: %s" % (
                backend, world, key, mode, ", ".join("%d pair(s) %.1f ms per block" % (
                    n, 1e3 * max(secs[((key, mode, cap, prec), n)]) / K) for n in PAIRS)))
    _RESULTS[(backend, world)] = {job: (refs[job], got[job]) for job, _, _ in jobs}
    return _RESULTS[(backend, world)]


@pytest.mark.parametrize("backend,world", TRANSPORTS)
@pytest.mark.parametrize("pairs", PAIRS)
@pytest.mark.parametrize("key,mode,cap,precision", CASES)
def test_sharded_get_async_equals_one_gpu_get(backend, world, pairs, key, mode, cap, precision):
    ref, ranks = _results(backend, world)[((key, mode, cap, precision), pairs)]
    for i in range(K):
        w = ref[i]
        rows = [r[i] for r in ranks]
        assert 1 < len(w["out"][0])
        if cap is not None:       # the cap cuts into the batch (and, with several ranks, into rank 1's shard)
            assert w["capped"] > 0
            assert sum(r["capped"] for r in rows) == w["capped"]
            if world > 1:
                assert rows[0]["capped"] > 0 and rows[1]["capped"] > 0
        root = rows[0]
        for f, (g, x) in enumerate(zip(root["out"], w["out"])):
            assert g.shape == x.shape and g.dtype == x.dtype, (i, f)
            if f in (2, 3):                               # adv, cadv
                np.testing.assert_allclose(g, x, rtol=2e-6, atol=2e-6, err_msg="%d %d" % (i, f))
            else:
                np.testing.assert_array_equal(g, x, err_msg="%d %d" % (i, f))
        # batch i is checked just before get_async() of batch i + 2; the last two have no such call
        assert root["intact"] is (True if i < K - 2 else None), i
        for r in rows[1:]:
            for (shape, dtype), x in zip(r["out"], w["out"]):
                assert shape == (0,) + x.shape[1:] and dtype == x.dtype
        for r in rows:
            assert r["bdiag"] == root["bdiag"] and r["diag"] == root["diag"]
            assert r["bdiag"]["poolm_batch_size"] == w["bdiag"]["poolm_batch_size"] == len(w["out"][0])
            for k in ("poolm_ret_mean", "poolm_cret_mean"):
                np.testing.assert_allclose(r["bdiag"][k], w["bdiag"][k], rtol=3e-7, atol=1e-9)
