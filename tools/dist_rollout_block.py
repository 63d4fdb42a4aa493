"""Time the model-rollout block of algorithms/cmbpo.py:241-270 sharded over G GPUs with ModelSampler.distribute():
archive sample (shard) -> reset -> sample(max_samples) loop -> finish_all_paths -> get() on rank 0.

    torchrun --nproc_per_node G tools/dist_rollout_block.py [--batches K] [--warmup W] [--pipelined] [--out FILE]

HCS, 7 x (512, 512) dynamics ensemble, 100 k start states in all, T = 35, schedule mode, fp16, max_samples = half of
B x 34 (the cap fires half way).  Prints one JSON line on rank 0: per batch, the whole block and get() on the root,
split into its device part (statistics, compaction, point-to-point receives) and its device->host copy; the bytes
each part moves; the card name and power limit read in the same run.

--pipelined: INTEGRATION.md's one-pair pipelined loop instead (reset / sample loop / finish_all_paths, get_async(),
result() of the previous batch), so that the root's device->host copy of batch i runs under the rollout of batch
i+1: wall time per batch over the timed batches, and the root's copy time from the device events of get_async()."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


class _ShapeEnv:
    class _S:
        def __init__(self, n):
            self.shape = (n,)

    def __init__(self, O, A):
        self.observation_space, self.action_space = self._S(O), self._S(A)


def _power_limit(dev):
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--B", type=int, default=100_000)
    ap.add_argument("--pipelined", action="store_true", help="time the pipelined loop with get_async()")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    dev = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(dev)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29531")
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", dev))
    try:
        import cmbpo_b200 as cb
        from cmbpo_b200 import _lib as L, workload as wl
        from cmbpo_b200.dist import shard_bounds
        task, O, A, B, T = "HalfCheetahSafe-v2", 17, 6, args.B, 35
        max_samples = B * (T - 1) // 2
        dyn, actor, v, vc = wl.make_problem(1, O, A, hidden=(512, 512), task=task)
        eng = cb.Engine(dev, precision="fp16")
        model = cb.B200PE.from_arrays(eng, L.NET_DYN, dyn)
        policy = cb.B200Policy(eng)
        policy.load_actor(actor.W, actor.b, actor.log_std)
        policy.load_values(v, vc)
        n_arch = 2 * B
        obs, _ = wl.make_states(2, n_arch, O, A, dyn)
        rng = np.random.default_rng(3)
        arch = cb.DeviceArchive(eng, n_arch, O, A, seed=4)
        arch.append(obs, (0.3 * rng.standard_normal((n_arch, A))).astype(np.float32),
                    np.broadcast_to(actor.log_std, (n_arch, A)).astype(np.float32),
                    np.repeat(np.arange(4, dtype=np.int32), n_arch // 4))
        env = cb.FakeEnv(_ShapeEnv(O, A), task, model, True, True, False)
        lo, hi = shard_bounds(B, rank, world)
        pool = cb.ModelBuffer(hi - lo, O, A, T, engine=eng)
        pool.initialize({"mu": (A,), "log_std": (A,)})
        smp = cb.ModelSampler(T, B, "schedule", seed=5)
        smp.initialize(env, policy, pool)
        smp.distribute()
        row_bytes = 4 * (O + A + 8 + A)                   # obs, act, 8 scalars, mu (log_std: one row)

        def rollout():
            start = arch.sample_start_states(policy, B, shard=(lo, hi))["observations"]
            smp.reset(start)
            while True:
                _, _, _, info = smp.sample(max_samples)
                if smp._total_samples >= 0.99 * max_samples or info["alive_ratio"] <= 0.0:
                    break
            smp.finish_all_paths()

        res = dict(world=world, B=B, T=T, max_samples=max_samples, precision="fp16",
                   api="get_async" if args.pipelined else "get")
        if args.pipelined:
            pending, copy_ms, rows_total = None, [], 0
            dist.barrier()
            for it in range(args.warmup + args.batches):
                if it == args.warmup:
                    t0 = time.perf_counter()
                rollout()
                handle = pool.get_async()
                if pending is not None:
                    host, diag = pending.result()
                    if rank == 0 and it > args.warmup:    # the copy of a timed batch
                        copy_ms.append(pending.copy_ms())
                    rows_total = diag["poolm_batch_size"]
                    del host
                pending = handle
            host, diag = pending.result()
            t1 = time.perf_counter()
            if rank == 0:
                copy_ms.append(pending.copy_ms())
            del host
            block = 1e3 * (t1 - t0) / args.batches
            res.update(rows_per_batch=int(rows_total), block_ms=block,
                       transitions_per_s=float(rows_total / (block * 1e-3)),
                       d2h_bytes=int(rows_total * row_bytes + 4 * A))
            if rank == 0:
                res.update(d2h_ms=float(np.median(copy_ms)),
                           d2h_GBps=float(rows_total * row_bytes / np.median(copy_ms) / 1e6))
        else:
            rows_total = rows_remote = 0
            block_ms, get_ms, get_dev_ms, d2h_ms = [], [], [], []
            for it in range(args.warmup + args.batches):
                torch.cuda.synchronize()
                dist.barrier()
                t0 = time.perf_counter()
                rollout()
                torch.cuda.synchronize()
                t1 = time.perf_counter()
                n_local = pool.size
                out, diag = pool.get_device()
                torch.cuda.synchronize()
                t2 = time.perf_counter()
                host = pool.to_host(out)
                pool.reset()
                t3 = time.perf_counter()
                if it >= args.warmup:
                    block_ms.append(1e3 * (t3 - t0))
                    get_ms.append(1e3 * (t3 - t1))
                    get_dev_ms.append(1e3 * (t2 - t1))
                    d2h_ms.append(1e3 * (t3 - t2))
                    rows_total = diag["poolm_batch_size"]
                    rows_remote = rows_total - (n_local if rank == 0 else 0)
                del host, out
            res.update(rows_per_batch=int(rows_total),
                       block_ms=float(np.median(block_ms)), get_ms=float(np.median(get_ms)),
                       transitions_per_s=float(rows_total / (np.median(block_ms) * 1e-3)),
                       get_device_ms=float(np.median(get_dev_ms)), get_d2h_ms=float(np.median(d2h_ms)),
                       p2p_bytes=int(rows_remote * row_bytes), d2h_bytes=int(rows_total * row_bytes + 4 * A),
                       d2h_GBps=float(rows_total * row_bytes / np.median(d2h_ms) / 1e6),
                       block_ms_all=[round(x, 3) for x in block_ms])
        res.update(gpu=torch.cuda.get_device_name(dev), power_limit=_power_limit(dev))
        all_res = [None] * world
        dist.all_gather_object(all_res, res)
        if rank == 0:
            line = json.dumps(dict(all_res[0], ranks_block_ms=[r["block_ms"] for r in all_res]))
            print(line)
            if args.out:
                with open(args.out, "a") as f:
                    f.write(line + "\n")
        eng.close()
    finally:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
