"""CPU: the batch-wide rules of a sharded rollout block (cmbpo_b200.dist, used by ModelSampler.distribute).

* cap_split: the max_samples cap of the reference cuts the first n surviving paths of the WHOLE batch by path
  index; with contiguous shards every rank cuts a prefix of its own survivors.  Checked against a brute force
  over random global path lists.
* all_gather_host + rank_order_sum over gloo: the gathered length histograms and per-step sums combine to the
  whole batch's, bit-identical on every rank."""
import os
import socket

import numpy as np
import torch.multiprocessing as mp

from cmbpo_b200.dist import cap_split, rank_order_sum, shard_bounds


def _brute_force(n, alive, sizes):
    """alive: survivor flag of every path of the batch (global order); returns the per-rank cut counts."""
    surviving = np.flatnonzero(alive)                 # ascending global path index
    cut = np.zeros(len(alive), bool)
    cut[surviving[:n]] = True
    starts = np.concatenate([[0], np.cumsum(sizes)])
    return [int(cut[starts[r]:starts[r + 1]].sum()) for r in range(len(sizes))]


def test_cap_split_matches_brute_force():
    rng = np.random.default_rng(0)
    for trial in range(3000):
        world = int(rng.integers(1, 9))
        sizes = rng.integers(0, 40, world)
        if trial % 5 == 0:
            sizes[rng.integers(0, world, max(1, world // 2))] = 0          # empty shards
        alive = rng.random(int(sizes.sum())) < rng.random()
        total = int(alive.sum())
        starts = np.concatenate([[0], np.cumsum(sizes)])
        survivors = [int(alive[starts[r]:starts[r + 1]].sum()) for r in range(world)]
        for n in {0, total, total + int(rng.integers(1, 5)), int(rng.integers(0, total + 1))}:
            got = cap_split(n, survivors)
            assert got == _brute_force(n, alive, sizes), (n, sizes, survivors)
            assert sum(got) == min(n, total)


def test_cap_split_edges():
    assert cap_split(0, [3, 4]) == [0, 0]
    assert cap_split(2, [3, 4]) == [2, 0]            # inside rank 0's shard
    assert cap_split(5, [3, 4]) == [3, 2]            # straddles ranks
    assert cap_split(99, [3, 0, 4]) == [3, 0, 4]     # more than all survivors
    assert cap_split(4, [0, 0, 5]) == [0, 0, 4]
    assert cap_split(3, []) == []


def test_rank_order_sum_is_sequential():
    g = np.array([[1e16, 1.0], [1.0, 2.0], [-1e16, 3.0]])
    np.testing.assert_array_equal(rank_order_sum(g), [(1e16 + 1.0) + -1e16, 6.0])
    h = np.arange(24, dtype=np.int64).reshape(4, 6)
    np.testing.assert_array_equal(rank_order_sum(h), h.sum(axis=0))


B, T = 1001, 9


def _batch():
    rng = np.random.default_rng(3)
    length = rng.integers(0, T + 1, B)
    uncertain = rng.random(B) < 0.3
    stats = rng.standard_normal((B, T)) * 3.0                         # per-path, per-step float64 values
    return length, uncertain, stats


def _local_tables(length, uncertain, stats):
    """What one rank reads from its shard: cmbpo_rollout_histogram's 2 (T + 1) int64 and step_stats[:, 0:2]."""
    h = np.concatenate([np.bincount(length, minlength=T + 1),
                        np.bincount(length[uncertain], minlength=T + 1)]).astype(np.int64)
    alive = np.arange(T)[None, :] < length[:, None]
    st = np.stack([alive.sum(0).astype(np.float64), np.where(alive, stats, 0.0).sum(0)], axis=1)
    return h, st


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, q):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from cmbpo_b200.dist import all_gather_host, rank_order_sum, shard_bounds
    length, uncertain, stats = _batch()
    lo, hi = shard_bounds(B, rank, world)
    h, st = _local_tables(length[lo:hi], uncertain[lo:hi], stats[lo:hi])
    gh = all_gather_host(h)
    gs = all_gather_host(np.ascontiguousarray(st))
    q.put((rank, gh, rank_order_sum(gh), rank_order_sum(gs)))
    dist.destroy_process_group()


def test_gathered_histograms_and_step_stats_combine_to_the_batch():
    world = 3
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=120) for _ in range(world)), key=lambda x: x[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    length, uncertain, stats = _batch()
    h_all, st_all = _local_tables(length, uncertain, stats)
    for rank, gh, h, st in res:
        lo, hi = shard_bounds(B, rank, world)
        assert gh.shape == (world, 2 * (T + 1))
        np.testing.assert_array_equal(gh[rank], _local_tables(length[lo:hi], uncertain[lo:hi], stats[lo:hi])[0])
        np.testing.assert_array_equal(h, h_all)                     # counts: exact
        np.testing.assert_array_equal(st[:, 0], st_all[:, 0])
        np.testing.assert_allclose(st[:, 1], st_all[:, 1], rtol=1e-12, atol=1e-12)
        # the same bits on every rank
        np.testing.assert_array_equal(h, res[0][2])
        assert st.tobytes() == res[0][3].tobytes()
