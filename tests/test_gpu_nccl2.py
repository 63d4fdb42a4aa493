"""-m gpu, needs >= 2 GPUs (skipped otherwise): two NCCL ranks, one per GPU, roll out the two halves of a batch
(weights broadcast from rank 0, Philox keyed by GLOBAL path id), run GAE, all-reduce the advantage statistics
and normalise; the gathered sample lists must equal the single-rank result of the whole batch: rows bit-exact
(paths are independent), normalised advantages equal because both sides use the same all-reduced float64 sums
up to the summation order of the two partial sums (tolerance 2 float32 ulp of the statistics)."""
import os
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

B, T, O, A = 3000, 12, 17, 6
GAE = dict(gamma=0.99, lam=0.95, cost_gamma=0.97, cost_lam=0.5)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _run_shard(eng, cb, L, wl, torch, nets, obs, lo, hi, reduce_fn, precision):
    dyn, actor, v, vc = nets
    n = hi - lo
    bufs = cb.RolloutBuffers(eng, n, T, O, A)
    bufs.set_inputs(obs[lo:hi])
    cfg = L.EnvCfg(L.TERM_NO_DONE, L.COST_HCS, 0, 1, 1)
    # uncertainty mode with a finite limit: ragged path lengths, so the gathered order matters
    bufs.run(cfg, uncertainty_mode=True, dkl_lim=_run_shard.dkl_lim, seed=77, path_id_base=lo, precision=precision)
    bufs.gae(GAE["gamma"], GAE["lam"], GAE["cost_gamma"], GAE["cost_lam"])
    sums = eng.adv_statistics_device(bufs.adv, bufs.cadv, bufs.ret, bufs.cret, n, T, 1, n, bufs.length, reduce_fn)
    eng.adv_normalise_device(bufs.adv, bufs.cadv, n, T, 1, n, bufs.length, sums)
    st = eng.stats_from_sums(sums.cpu().numpy())
    torch.cuda.synchronize()
    out = {k: bufs.host(k) for k in ("obs", "act", "nextobs", "rew", "val", "cval", "cost", "logp", "adv", "cadv", "ret", "cret")}
    out["length"] = bufs.length.cpu().numpy()
    out["stats"] = np.array([st["n"], st["adv_mean"], st["adv_std"], st["cadv_mean"]], np.float64)
    return out


def _load(eng, cb, L, nets, torch, dist, dev, bcast):
    dyn, actor, v, vc = nets

    def b(a):
        x = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
        if bcast:
            if dist.get_rank() != 0:
                x.zero_()                      # only rank 0's weights survive: proves the broadcast is what loads them
            dist.broadcast(x, 0)
        return x

    for which, en, prob in ((L.NET_DYN, dyn, True), (L.NET_V, v, False), (L.NET_VC, vc, False)):
        eng.set_network(which, [b(w) for w in en.W], [b(x) for x in en.b], en.acts, b(en.mu_in), b(en.var_in),
                        b(en.mu_out), b(en.var_out), prob, en.elite_inds)
    eng.set_actor([b(w) for w in actor.W], [b(x) for x in actor.b], b(actor.log_std))


def _worker(rank, world, port, precision, dkl_lim, q):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L, workload as wl
    from cmbpo_b200.dist import shard_bounds, make_reduce_fn
    nets = wl.make_problem(3, O, A, hidden=(512, 512))
    obs, _ = wl.make_states(4, B, O, A, nets[0])
    eng = cb.Engine(rank, precision=precision)
    _load(eng, cb, L, nets, torch, dist, dev, bcast=True)
    lo, hi = shard_bounds(B, rank, world)
    _run_shard.dkl_lim = dkl_lim
    out = _run_shard(eng, cb, L, wl, torch, nets, obs, lo, hi, make_reduce_fn(), precision)
    q.put((rank, lo, hi, out))
    dist.barrier()
    dist.destroy_process_group()
    eng.close()


@pytest.mark.parametrize("precision", ["fp16", "fp32"])
def test_two_nccl_ranks_equal_one_rank(precision):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    import cmbpo_b200 as cb
    from cmbpo_b200 import _lib as L, workload as wl
    nets = wl.make_problem(3, O, A, hidden=(512, 512))
    obs, _ = wl.make_states(4, B, O, A, nets[0])
    # single rank, whole batch
    eng = cb.Engine(0, precision=precision)
    _load(eng, cb, L, nets, torch, None, torch.device("cuda", 0), bcast=False)
    # a limit that cuts a good share of the paths: 6 x the mean one-step disagreement
    one = eng.fakeenv_step(L.EnvCfg(L.TERM_NO_DONE, L.COST_HCS, 0, 1, 1), obs, np.zeros((B, A), np.float32), seed=1)
    dkl_lim = 6.0 * float(one["dkl_mean"].item())
    _run_shard.dkl_lim = dkl_lim
    ref = _run_shard(eng, cb, L, wl, torch, nets, obs, 0, B, None, precision)
    eng.close()
    assert 1 < ref["length"].mean() < T - 1, "the limit should produce ragged paths"

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, precision, dkl_lim, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=300) for _ in range(2)), key=lambda x: x[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert res[0][1] == 0 and res[0][2] == res[1][1] and res[1][2] == B
    # every rank derived the same global statistics, equal to the one-rank ones
    np.testing.assert_array_equal(res[0][3]["stats"], res[1][3]["stats"])
    assert res[0][3]["stats"][0] == ref["stats"][0]
    np.testing.assert_allclose(res[0][3]["stats"][1:], ref["stats"][1:], rtol=3e-7, atol=1e-9)
    # gathered rows (rank order = path order) are the one-rank rows, bit for bit
    for k in ("length", "obs", "act", "nextobs", "rew", "val", "cval", "cost", "logp", "ret", "cret"):
        got = np.concatenate([res[0][3][k], res[1][3][k]], axis=0)
        np.testing.assert_array_equal(got, ref[k], err_msg=k)
    for k in ("adv", "cadv"):
        got = np.concatenate([res[0][3][k], res[1][3][k]], axis=0)
        np.testing.assert_allclose(got, ref[k], rtol=2e-6, atol=2e-6, err_msg=k)
