#!/usr/bin/env python
"""bench.py -- model-rollout transitions/sec (+ GAE ms per 1M steps) of the CMBPO hot path.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # CPU: the oracle port of the reference
    python bench.py ... --dump-outputs DIR                    # + the last timed step's outputs as DIR/<name>.npy

One "step" = one pass of the hot path over one batch of synthetic start states:
H-step model rollout (policy -> PENS ensemble -> FakeEnv statics -> ModelBuffer write-out), GAE +
cost-GAE scans, advantage statistics / normalisation.  Workload at every N: BASELINE.json
configs[1] -- HalfCheetahSafe (obs 17, act 6), 7x(512,512) swish ensemble, 100 000 start states per
GPU, maxroll 35 (34 stored steps), deterministic-mean transitions, Philox noise; weak scaling
(start states sharded across ranks, no data-path collective, one tiny all-reduce of statistics).
Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

if "reference" in sys.argv and int(os.environ.get("RANK", "0")) == 0:
    # the reference arm runs on rank 0 alone with ALL host threads; torchrun pins OMP_NUM_THREADS=1
    # for its children, which must be undone before numpy loads its BLAS
    for _k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
        os.environ[_k] = str(len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else os.cpu_count())

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TASK, OBS, ACT = "HalfCheetahSafe-v2", 17, 6
HIDDEN, E = (512, 512), 7
MAXROLL = 35
GAE = dict(gamma=0.99, lam=0.95, cost_gamma=0.97, cost_lam=0.5)
METRIC, UNIT = "model-rollout transitions/sec", "transitions/s"
WORKLOAD = ("BASELINE configs[1]: HalfCheetahSafe H-step model rollout + GAE/cost-GAE + advantage normalisation")
# BASELINE.json configs[1..4] (SURVEY.md section 8d); the default line is configs[1]
TASKS = {"hcs": ("HalfCheetahSafe-v2", 17, 6), "ant": ("AntSafe-v2", 29, 8), "hum": ("HumanoidSafe-v2", 47, 17)}
CONFIGS = {
    "hcs": dict(task="hcs", workload=WORKLOAD, scaling="weak"),
    "ant1m": dict(task="ant", scaling="strong", total=1000000,
                  workload="BASELINE configs[2]: AntSafe ensemble rollout, 1M start states sharded over the ranks "
                           "(termination function shortens paths; alive-row compaction) + GAE/cost-GAE + normalisation"),
    "hcs_unc": dict(task="hcs", scaling="weak", total_per_gpu=100000,
                    workload="HalfCheetahSafe H-step rollout in the reference's DEFAULT rollout_mode 'uncertainty' "
                             "(configs/cmbpo_hcs.py:28): a path is cut when its cumulative ensemble KL reaches dkl_lim = "
                             "rollout_schedule[2] (= 5) x the mean one-step KL of 5000 start states (cmbpo.py:198-200); "
                             "alive-row compaction; + GAE/cost-GAE + normalisation"),
    "hs_gae": dict(task="hum", scaling="weak",
                   workload="BASELINE configs[3]: HumanoidSafe (configs/cmbpo_hs) rollout feeding the GAE + cost-GAE "
                            "reverse scans; standalone GAE layouts in `gae_layouts`"),
    "sweep": dict(task="hcs", scaling="strong",
                  workload="BASELINE configs[4]: HalfCheetahSafe roofline sweep, horizon H x total start states B "
                           "(sharded over the ranks)"),
}


_REAL_STDOUT = None


def emit(line):
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(line), flush=True)


def host_threads():
    """Threads the numpy BLAS behind the oracle port actually uses (what `cores` reports)."""
    try:
        from threadpoolctl import threadpool_info
        n = [p.get("num_threads", 0) for p in threadpool_info() if p.get("user_api") == "blas"]
        if n:
            return int(max(n))
    except Exception:
        pass
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def flop_per_transition(O=OBS, A=ACT, h=HIDDEN[0]):
    """BASELINE.md section 3: dynamics + actor + V,VC, un-padded dims."""
    D, Din = O + 1, O + A
    dyn = 2 * E * (Din * h + h * h + h * 2 * D)
    actor = 2 * (O * 128 + 128 * 128 + 128 * A)
    vvc = 2 * 3 * 2 * (O * 128 + 128 * 128 + 128)
    return dyn, actor, vvc


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sus=p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                    src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sus=1400.0, src="fallback")


def ncu_traffic():
    """DRAM bytes per launch of K1 from the committed `ncu --set full` summary (profiles/), or None."""
    for name in ("r2_k1_traffic.json", "r1_k1_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                return json.load(f)["dram_bytes_per_launch"]
        except Exception:
            continue
    return None


def ncu_tensor_pipe():
    """sm__pipe_tensor_cycles_active (% of elapsed) of K1 from the committed ncu summary, or None."""
    for name in ("r2_k1_ncu.txt", "r1_k1_ncu.txt"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                for ln in f:
                    if ln.startswith("sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed"):
                        return {"value": float(ln.split()[-1].replace(",", "")), "source": "profiles/" + name}
        except Exception:
            continue
    return None


def bind_to_gpu_numa_node(local_rank):
    """Pin this rank's process to the CPU cores NVML reports as local to its GPU, so that page-locked host buffers
    (first touched by this process) and the D2H copies stay on the GPU's NUMA node.  Returns the core count or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = local_rank
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if local_rank < len(ids) and ids[local_rank].isdigit():
                phys = int(ids[local_rank])
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        n_words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = {w * 64 + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


class ClockSampler:
    """SM clock / power / throttle reasons sampled DURING the timed region (B200_PROFILING.md's clocks
    line), through NVML in a thread (initialised before the region starts: spawning nvidia-smi takes
    longer than a short timed region on an 8-GPU box); falls back to `nvidia-smi -lms`."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.proc, self.lines = gpu_index, None, []
        self.nvml, self.handle, self.samples, self.stop_flag = None, None, [], False

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # LOCAL_RANK indexes the visible devices; map through CUDA_VISIBLE_DEVICES when it is a list of indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = self.idx
            if vis:
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if self.idx < len(ids) and ids[self.idx].isdigit():
                    phys = int(ids[self.idx])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                pw = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
                rs = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)) if hasattr(n, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                self.samples.append((sm, pw, rs))
            except Exception:
                pass
            time.sleep(0.02)

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=1)
            if not self.samples:
                return {"sm_mhz": None, "sm_max_mhz": self.max_sm, "reasons": ["no samples"]}
            n = self.nvml
            bits = {"hw_slowdown": getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                    "hw_thermal_slowdown": getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                    "sw_thermal_slowdown": getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                    "sw_power_cap": getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
            reasons = sorted(k for k, b in bits.items() if any(r & b for _, _, r in self.samples))
            pmax = max(p for _, p, _ in self.samples)
            load = [s for s, p, _ in self.samples if p > 0.5 * pmax] or [s for s, _, _ in self.samples]
            return {"sm_mhz": float(np.median(load)), "sm_max_mhz": self.max_sm, "power_w_max": float(pmax),
                    "samples": len(self.samples), "reasons": reasons, "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        load = [s for s, p in zip(sm, power) if p > 0.5 * max(power)] or sm
        return {"sm_mhz": float(np.median(load)), "sm_max_mhz": float(max(mx)),
                "power_w_max": float(max(power)), "samples": len(sm), "reasons": sorted(reasons),
                "source": "nvidia-smi"}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference (numpy), bounded sample of the same workload
# ------------------------------------------------------------------------------------------------
def cpu_rollout_sample(B, seed=0):
    """One reference-port pass (reset -> sample x 34 -> finish_all_paths -> get) on B start states."""
    from oracle import cmbpo_oracle as orc
    orc.FAST_GEMM = True      # the member contraction as one multi-threaded BLAS GEMM (timing legs only)
    dyn, actor, v, vc = orc.make_problem(seed, OBS, ACT, hidden=HIDDEN, task=TASK)
    obs, _ = orc.make_states(seed + 1, B, OBS, ACT, dyn)
    noise = orc.TableNoise(seed + 2, MAXROLL, B, ACT, len(dyn.elite_inds))
    t0 = time.perf_counter()
    out, bdiag, diag, _ = orc.run_rollout(dyn, actor, v, vc, TASK, obs, noise, MAXROLL,
                                          gamma=GAE["gamma"], lam=GAE["lam"],
                                          cgamma=GAE["cost_gamma"], clam=GAE["cost_lam"])
    dt = time.perf_counter() - t0
    return len(out[0]), dt


def cpu_single_step(n_rows, seed=0):
    """BASELINE configs[0]: one FakeEnv.step (predict_ensemble + average_dkl + statics) on n_rows synthetic
    (obs17, act6) rows through the oracle port; rows per second."""
    from oracle import cmbpo_oracle as orc
    orc.FAST_GEMM = True      # the member contraction as one multi-threaded BLAS GEMM (timing legs only)
    dyn, actor, v, vc = orc.make_problem(seed, OBS, ACT, hidden=HIDDEN, task=TASK)
    obs, act = orc.make_states(seed + 1, n_rows, OBS, ACT, dyn)
    noise = orc.TableNoise(seed + 2, 2, n_rows, ACT, len(dyn.elite_inds))
    env = orc.OracleFakeEnv(OBS, ACT, TASK, orc.OracleModel(dyn), noise.idx_fn)
    env.ctx = (0, np.arange(256))
    env.step(obs[:256], act[:256])
    env.ctx = (0, np.arange(n_rows))
    t0 = time.perf_counter()
    env.step(obs, act)
    dt = time.perf_counter() - t0
    return n_rows / dt, dt


def cpu_gae_ms_per_1m():
    from oracle import cmbpo_oracle as orc
    orc.FAST_GEMM = True      # the member contraction as one multi-threaded BLAS GEMM (timing legs only)
    rng = np.random.default_rng(0)
    B, T = 8192, 34
    r, v, c, cv = (rng.standard_normal((B, T)).astype(np.float32) for _ in range(4))
    lv, lc = (rng.standard_normal(B).astype(np.float32) for _ in range(2))
    t0 = time.perf_counter()
    orc.gae_path(r, v, c, cv, lv, lc, 0.99, 0.95, 0.97, 0.5)
    return (time.perf_counter() - t0) * 1e3 / (B * T / 1e6)


def cpu_gae_reference_ms_per_1m():
    """BASELINE.md B4: the reference's GAE arithmetic on the host -- `np.append`, deltas, flip /
    `scipy.signal.lfilter([1],[1,-d])` / flip (utilities/utils.py:186-188 as called by modelbuffer.py:163-179), float64
    output stored into float32 buffers -- over 1 M steps as [32768 paths x 32 steps] and as one flat CPOBuffer of
    1049 paths x 1000 steps (one `finish_path` per path, cpobuffer.py:179-207).  scipy is single threaded."""
    import scipy.signal
    rng = np.random.default_rng(0)

    def gae(r, v, c, cv, lv, lc):
        out = []
        for x, val, last, g, lam in ((r, v, lv, 0.99, 0.95), (c, cv, lc, 0.97, 0.5)):
            vals = np.append(val, last, axis=-1)
            deltas = x + g * vals[..., 1:] - vals[..., :-1]
            flipped = np.flip(deltas, axis=-1)
            adv = np.flip(scipy.signal.lfilter([1], [1, float(-g * lam)], flipped, axis=-1), axis=-1).astype(np.float32)
            out += [adv, (adv + val).astype(np.float32)]
        return out

    B, T = 32768, 32
    r, v, c, cv = (rng.standard_normal((B, T)).astype(np.float32) for _ in range(4))
    lv, lc = (rng.standard_normal((B, 1)).astype(np.float32) for _ in range(2))
    gae(r[:64], v[:64], c[:64], cv[:64], lv[:64], lc[:64])
    t0 = time.perf_counter()
    gae(r, v, c, cv, lv, lc)
    batched = (time.perf_counter() - t0) * 1e3 / (B * T / 1e6)
    P, L_ = 1049, 1000
    r, v, c, cv = (rng.standard_normal(P * L_).astype(np.float32) for _ in range(4))
    t0 = time.perf_counter()
    for i in range(P):
        sl = slice(i * L_, (i + 1) * L_)
        gae(r[sl], v[sl], c[sl], cv[sl], np.zeros(1, np.float32), np.zeros(1, np.float32))
    flat = (time.perf_counter() - t0) * 1e3 / (P * L_ / 1e6)
    return {"paths_32768x32_ms_per_1M_steps": batched, "flat_1049x1000_ms_per_1M_steps": flat,
            "what": "BASELINE.md B4: scipy.signal.lfilter GAE + cost-GAE exactly as the reference calls it, one host thread"}


def cpu_single_step_torch(n_rows, seed=0):
    """BASELINE.md B2: the same single FakeEnv.step with the three ensemble GEMMs through torch-CPU `bmm` (MKL, all
    threads) instead of numpy; the head / KL / statics arithmetic stays the oracle port's.  rows per second."""
    import torch
    from oracle import cmbpo_oracle as orc
    orc.FAST_GEMM = True      # the member contraction as one multi-threaded BLAS GEMM (timing legs only)
    dyn, actor, v, vc = orc.make_problem(seed, OBS, ACT, hidden=HIDDEN, task=TASK)
    obs, act = orc.make_states(seed + 1, n_rows, OBS, ACT, dyn)
    W = [torch.from_numpy(np.ascontiguousarray(w)) for w in dyn.W]
    bs = [torch.from_numpy(np.ascontiguousarray(np.asarray(b).reshape(w.shape[0], 1, -1))) for w, b in zip(dyn.W, dyn.b)]
    sig_in = torch.from_numpy(np.maximum(np.sqrt(dyn.var_in), 1e-2).astype(np.float32))
    mu_in = torch.from_numpy(np.asarray(dyn.mu_in, np.float32))

    def forward(x):
        h = ((torch.from_numpy(x) - mu_in) / sig_in).unsqueeze(0).expand(W[0].shape[0], -1, -1)
        for i, (w, b) in enumerate(zip(W, bs)):
            h = torch.baddbmm(b, h, w)
            if i < len(W) - 1:
                h = h * torch.sigmoid(h)
        return h.numpy()

    x = np.concatenate([obs, act], -1).astype(np.float32)
    forward(x[:256])
    t0 = time.perf_counter()
    raw = forward(x)
    D = raw.shape[-1] // 2
    sig_o = np.maximum(np.sqrt(dyn.var_out), 1e-2).astype(np.float32)
    mean = raw[..., :D] * sig_o + dyn.mu_out
    var = np.exp(raw[..., D:] + 2 * np.log(sig_o))
    std = np.sqrt(var)
    orc.average_dkl(mean[..., :OBS], std[..., :OBS]).mean(-1)
    np.var(mean[..., :OBS], axis=0)
    orc.hcs_cost(mean[0, :, :OBS] + obs)
    dt = time.perf_counter() - t0
    return n_rows / dt, dt, int(torch.get_num_threads())


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = host_threads()
    B = args.cpu_batch
    for _ in range(args.warmup):                      # W warm-up passes (small: BLAS thread pools, page faults)
        cpu_rollout_sample(min(B, 200))
    times, n_tr = [], 0
    for s in range(args.steps):
        n, dt = cpu_rollout_sample(B, seed=s)
        times.append(dt); n_tr += n
    total = sum(times)
    value = n_tr / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "impl_note": "CPU port of the reference (numpy restatement of the TF "
                               "graphs; TF 1.14 is not installable; ensemble contractions as multi-threaded BLAS GEMMs), bounded sample of the workload per step",
                   "start_states_per_step": B, "maxroll": MAXROLL, "stored_steps": MAXROLL - 1, "obs": OBS,
                   "act": ACT, "ensemble": "7x(512,512) swish, 5 elites"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d start states x %d steps per pass, %d passes" % (B, MAXROLL - 1, args.steps),
                         "gae_ms_per_1M_steps": cpu_gae_ms_per_1m(), "gae": cpu_gae_reference_ms_per_1m()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------------
# CUDA arm
# ------------------------------------------------------------------------------------------------
DUMP_BYTES = 48 << 20      # budget of the sampled per-path fields of --dump-outputs (the whole dump stays below 64 MB)


def dump_outputs(out_dir, bufs, sums):
    """--dump-outputs: what the last timed pass leaves for its caller, as <out_dir>/<name>.npy in float32 / float64.
    `adv_stats_sums` are the 8 float64 advantage-statistics sums of the whole batch (all ranks).  Every per-step and
    per-path field of the rollout buffers is written for a fixed sample of paths (seed 0, listed in `path_index`,
    as many as fit DUMP_BYTES) in the reference's [path, step, ...] layout, with the steps at or past a path's
    length zeroed: they are not part of its sample list.  Integer fields are written as float32 (exact: small)."""
    import torch
    from cmbpo_b200.rollout import STEP_FIELDS_VEC, STEP_FIELDS, GAE_FIELDS
    step_fields = STEP_FIELDS_VEC + STEP_FIELDS + GAE_FIELDS + ("term",)
    path_fields = ("length", "end_reason", "last_val", "last_cval", "cum_dkl", "final_obs")
    path_bytes = sum(bufs.T * getattr(bufs, f)[0, 0].numel() * 4 for f in step_fields) + \
        sum(getattr(bufs, f)[0].numel() * 8 for f in path_fields)
    n = min(bufs.B, DUMP_BYTES // path_bytes)
    idx = np.sort(np.random.default_rng(0).choice(bufs.B, n, replace=False))
    sel = torch.from_numpy(idx).to(bufs.length.device)
    alive = torch.arange(bufs.T, device=sel.device)[None, :] < bufs.length.index_select(0, sel).long()[:, None]
    out = {"path_index": torch.from_numpy(idx.astype(np.float64)), "adv_stats_sums": sums}
    for f in step_fields:
        x = getattr(bufs, f).index_select(1, sel).transpose(0, 1)           # time-major [T, B, ...] -> [n, T, ...]
        out[f] = torch.where(alive if x.dim() == 2 else alive[..., None], x, torch.zeros((), dtype=x.dtype, device=x.device))
    for f in path_fields:
        out[f] = getattr(bufs, f).index_select(0, sel)
    os.makedirs(out_dir, exist_ok=True)
    for name, x in out.items():
        a = x.cpu().numpy()
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float32)
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


class Rig:
    """One rank's engine with the synthetic networks of a task shape loaded (weights generated on rank 0 and
    broadcast once over NCCL, then uploaded from device memory)."""

    def __init__(self, task_key, args, rank, world, local_rank):
        import torch
        import torch.distributed as dist
        import cmbpo_b200 as cb
        from cmbpo_b200 import _lib as L
        from cmbpo_b200 import workload as wl
        self.torch, self.dist, self.cb, self.L, self.wl = torch, dist, cb, L, wl
        self.rank, self.world, self.local_rank, self.args = rank, world, local_rank, args
        self.task, self.O, self.A = TASKS[task_key]
        self.dev = torch.device("cuda", local_rank)
        self.eng = cb.Engine(local_rank, precision=args.precision)
        self.unc_mode, self.dkl_lim = False, 0.0
        self.dyn, self.actor, self.v, self.vc = wl.make_problem(0, self.O, self.A, hidden=HIDDEN, task=self.task)
        dev = self.dev

        def bcast(a):
            x = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
            if world > 1:
                if rank != 0:
                    x.zero_()
                dist.broadcast(x, 0)
            return x

        def ens_dev(en):
            return dict(W=[bcast(w) for w in en.W], b=[bcast(b) for b in en.b], mu_in=bcast(en.mu_in),
                        var_in=bcast(en.var_in), mu_out=bcast(en.mu_out), var_out=bcast(en.var_out))

        self.dev_nets = {L.NET_DYN: ens_dev(self.dyn), L.NET_V: ens_dev(self.v), L.NET_VC: ens_dev(self.vc)}
        self.dev_actor = ([bcast(w) for w in self.actor.W], [bcast(b) for b in self.actor.b], bcast(self.actor.log_std))
        self.load_engine(self.eng)
        term = L.TERM_ANTSAFE if task_key == "ant" else L.TERM_NO_DONE
        cost = {"hcs": L.COST_HCS, "ant": L.COST_ANTSAFE, "hum": L.COST_ZERO}[task_key]
        # --mode mean: deterministic-mean transitions (what ModelSampler runs, model_sampler.py:259);
        # --mode injected: mean + std * eps with Philox eps per (path, step, dim) (SURVEY.md 8a-Q1)
        self.env_cfg = L.EnvCfg(term, cost, 0, 0 if args.mode == "injected" else 1, 1)

    def load_engine(self, e):
        L = self.L
        for which, en, prob in ((L.NET_DYN, self.dyn, True), (L.NET_V, self.v, False), (L.NET_VC, self.vc, False)):
            d = self.dev_nets[which]
            e.set_network(which, d["W"], d["b"], en.acts, d["mu_in"], d["var_in"], d["mu_out"],
                          d["var_out"], prob, en.elite_inds)
        e.set_actor(*self.dev_actor)

    def reduce_fn(self, x):
        if self.world > 1:
            self.dist.all_reduce(x)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def flops(self, h=HIDDEN[0]):
        O, A = self.O, self.A
        D, Din = O + 1, O + A
        dyn = 2 * E * (Din * h + h * h + h * 2 * D)
        actor = 2 * (O * 128 + 128 * 128 + 128 * A)
        vvc = 2 * 3 * 2 * (O * 128 + 128 * 128 + 128)
        return dyn, actor, vvc

    def row_bytes(self):
        return (2 * self.O + 3 * self.A + 6) * 4 + 2          # SURVEY.md 8d: write-out bytes per stored transition

    def timed_rollouts(self, B, T, steps, warmup, seed0=1234, with_stats=True, dump=True):
        """`steps` passes of rollout -> GAE -> statistics -> normalise over B device-resident start states; with
        --dump-outputs and `dump`, rank 0 then writes the outputs of the last pass.
        Returns dict(ms, n_tr (whole job), launches, dyn_launch_ms, gae_launch_ms, breakdown, clocks)."""
        torch, eng, L = self.torch, self.eng, self.L
        obs_host, _ = self.wl.make_states(100 + self.rank, B, self.O, self.A, self.dyn)
        start = torch.from_numpy(obs_host).to(self.dev)
        bufs = self.cb.RolloutBuffers(eng, B, T, self.O, self.A)
        path_base = self.rank * B
        world = self.world

        def hot_path(step):
            bufs.start_obs = start
            bufs.run(self.env_cfg, seed=seed0 + step, path_id_base=path_base, precision=self.args.precision,
                     flags=(L.ROLLOUT_FUSE if self.args.fuse else 0), uncertainty_mode=self.unc_mode, dkl_lim=self.dkl_lim)
            bufs.gae(GAE["gamma"], GAE["lam"], GAE["cost_gamma"], GAE["cost_lam"])
            sums = eng.adv_statistics_device(bufs.adv, bufs.cadv, bufs.ret, bufs.cret, B, T, 1, B, bufs.length,
                                             self.reduce_fn if world > 1 else None)
            eng.adv_normalise_device(bufs.adv, bufs.cadv, B, T, 1, B, bufs.length, sums)
            return sums

        for w in range(warmup):
            hot_path(-1 - w)
        self.barrier()
        eng.profile(True)
        for k in range(4):
            eng.profile_read(k, True)
        clocks = ClockSampler(self.local_rank)
        clocks.start()
        launches0 = eng.launch_count
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        ev0.record()
        n_acc = torch.zeros(1, device=self.dev, dtype=torch.float64)
        for s_ in range(steps):
            sums = hot_path(s_)
            n_acc += sums[0:1]            # with N > 1 the statistics are all-reduced: already the whole-job count
        ev1.record()
        self.barrier()
        clk = clocks.stop()
        ms = ev0.elapsed_time(ev1)
        n_tr = float(n_acc.item())
        res = dict(ms=ms, n_tr=n_tr, launches=eng.launch_count - launches0, clocks=clk, obs_host=obs_host)
        for name, k in (("dyn", L_PROF_DYN), ("gae", L_PROF_GAE), ("step", 2), ("pol", 3)):
            t_ms, n = eng.profile_read(k, True)
            res[name + "_ms"], res[name + "_n"] = t_ms, n
        eng.profile(False)
        if dump and self.args.dump_outputs and self.rank == 0:
            dump_outputs(self.args.dump_outputs, bufs, sums)
        del bufs
        return res

    def reduce_result(self, res, extra_max=(), extra_sum=()):
        """max over ranks of the times, sum of the counts"""
        torch = self.torch
        vec = torch.tensor([res["ms"], res["dyn_ms"] / max(res["dyn_n"], 1), res["gae_ms"] / max(res["gae_n"], 1)] + list(extra_max),
                           device=self.dev, dtype=torch.float64)
        cnt = torch.tensor([res["n_tr"], res["launches"]] + list(extra_sum), device=self.dev, dtype=torch.float64)
        if self.world > 1:
            self.dist.all_reduce(vec, op=self.dist.ReduceOp.MAX)
            self.dist.all_reduce(cnt, op=self.dist.ReduceOp.SUM)
            cnt[0] /= self.world          # n_tr was global on every rank
        return [float(x) for x in vec], [float(x) for x in cnt]


def roofline_obj(pk, flop_per_row, rows_per_launch, launch_ms, step_ms, launches_per_pass, kernel_name):
    ach = flop_per_row * rows_per_launch / (launch_ms * 1e-3) / 1e12 if launch_ms > 0 else 0.0
    tp = ncu_tensor_pipe()
    return {"bound": "tensor", "kernel": kernel_name, "achieved": ach, "peak": pk["tf_burst"], "unit": "TFLOP/s",
            "frac": ach / pk["tf_burst"], "frac_burst": ach / pk["tf_burst"], "frac_sustained": ach / pk["tf_sus"],
            "peak_sustained": pk["tf_sus"],
            "peak_note": "%s bf16 GEMM peaks of MEASURED_PEAKS.json; `frac` is against the BURST figure (the timed "
                         "region is < 1 s at full clocks), frac_sustained against the 4 s / power-capped one" % pk["src"],
            "tensor_pipe_active_pct_ncu": tp, "traffic": ncu_traffic(),
            "launch_ms": launch_ms, "rows_per_launch": rows_per_launch, "flop_per_row": flop_per_row,
            "share_of_step": launch_ms * launches_per_pass / step_ms if step_ms > 0 else None}


def dtype_name(precision):
    return {"fp32": "f32", "fp16": "f16 (tcgen05 kind::f16, f32 accumulate)",
            "bf16": "bf16 (tcgen05 kind::f16, f32 accumulate)"}[precision]


def mode_name(args):
    return ("injected-noise (mean + std*eps, Philox eps)" if args.mode == "injected" else "deterministic-mean") + \
        ", Philox action noise / elite draws, " + ("uncertainty cut-off (see workload)" if args.config == "hcs_unc" else "dkl_lim=inf")


def run_cuda(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    args.numa_cores = bind_to_gpu_numa_node(local_rank) if world > 1 and not args.no_numa_bind else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    cfg = CONFIGS[args.config]
    rig = Rig(cfg["task"], args, rank, world, local_rank)
    try:
        {"hcs": bench_hcs, "ant1m": bench_ant1m, "hs_gae": bench_hs_gae, "sweep": bench_sweep,
         "hcs_unc": bench_hcs_unc}[args.config](rig, args, cfg)
    finally:
        if world > 1:
            dist.destroy_process_group()
        rig.eng.close()


def base_line(rig, args, cfg, value, ms_per_step, extra_config):
    c = {"workload": cfg["workload"], "maxroll": MAXROLL, "stored_steps": MAXROLL - 1, "obs": rig.O, "act": rig.A,
         "ensemble": "7x(512,512) swish, 5 elites", "policy": "tanh 128-128 + 2x(3x swish 128-128-1)",
         "mode": mode_name(args), "precision": args.precision,
         "step": "fused (CMBPO_ROLLOUT_FUSE: 2 launches per step)" if args.fuse else "step-wise (4 launches per step)"}
    c.update(extra_config)
    return {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": rig.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": cfg["scaling"],
            "vs_baseline": None, "dtype": dtype_name(args.precision), "data": "synthetic", "config": c}


# ---- configs[1]: the default line ----------------------------------------------------------------
def bench_hcs(rig, args, cfg):
    torch, cb, L, eng = rig.torch, rig.cb, rig.L, rig.eng
    world, rank, dev = rig.world, rig.rank, rig.dev
    B, T = args.batch, MAXROLL
    res = rig.timed_rollouts(B, T, args.steps, args.warmup)
    obs_host = res["obs_host"]
    path_base = rank * B

    # ---- end to end through the public API: host start states in, host sample list out ----
    class _Space:
        def __init__(self, n):
            self.shape = (n,)

    class ShapeEnv:
        observation_space, action_space = _Space(rig.O), _Space(rig.A)

    def make_pair(k):
        stream = torch.cuda.current_stream(dev) if k == 0 else torch.cuda.Stream(device=dev)
        with torch.cuda.stream(stream):
            e = eng if k == 0 else cb.Engine(rig.local_rank, precision=args.precision)
            if k:
                rig.load_engine(e)
            policy = cb.B200Policy(e)
            policy.attach_loaded(rig.actor.log_std)
            fenv = cb.FakeEnv(ShapeEnv(), rig.task, cb.B200PE.view(e, L.NET_DYN), True, True, False)
            pool = cb.ModelBuffer(B, rig.O, rig.A, T, engine=e)
            pool.initialize({"mu": (rig.A,), "log_std": (rig.A,)}, **GAE)
            pool.reduce_fn = rig.reduce_fn if world > 1 else None
            smp = cb.ModelSampler(T, B, False, logger=object(), seed=7 + k)
            smp.path_id_base = path_base
            smp.initialize(fenv, policy, pool)
        return smp, pool, stream

    def d2h_bytes(out):
        # bytes that crossed PCIe: a stride-0 axis (log_std, one row broadcast) is not copied
        return sum(int(np.prod([m for m, st in zip(a.shape, a.strides) if st != 0] or [1])) * a.itemsize for a in out)

    # (1) `e2e`: the unmodified caller's sequence (algorithms/cmbpo.py:251-269): reset -> sample until the alive
    # ratio drops -> finish_all_paths -> get(), one sampler / buffer pair, blocking get() that returns caller-owned
    # numpy arrays.
    def plain_batch(pair):
        smp, pool, _ = pair
        smp.reset(obs_host)
        while True:
            _, _, _, info = smp.sample(None)
            if info["alive_ratio"] <= 0.1:
                break
        smp.finish_all_paths()
        out, _ = pool.get()
        return out

    # (2) `e2e_pipelined`: two sampler / buffer pairs, each on its own engine (= its own CUDA stream), used
    # alternately: reset() only queues the rollout, so batch i+1 rolls out while the host walks batch i through
    # sample() / finish_all_paths() / get_async() and while the device->host copy of batch i runs on a side
    # stream.  get_async() is an extension of the reference interface; its arrays are views of recycled
    # page-locked buffers (valid until the second next get_async of that buffer).
    def e2e_reset(pairs, k):
        with torch.cuda.stream(pairs[k][2]):
            pairs[k][0].reset(obs_host)              # H2D of the start states, rollout queued

    def e2e_collect(pairs, k):
        smp, pool, stream = pairs[k]
        with torch.cuda.stream(stream):
            while True:
                _, _, _, info = smp.sample(None)    # the first call waits for this pair's rollout
                if info["alive_ratio"] <= 0.1:
                    break
            smp.finish_all_paths()
            return pool.get_async()

    def pipelined_run(pairs, n_batches):
        n, handles, out = 0, [], None
        e2e_reset(pairs, 0)
        for i in range(n_batches):
            if i + 1 < n_batches:
                e2e_reset(pairs, (i + 1) & 1)
            handles.append(e2e_collect(pairs, i & 1))
            if len(handles) == 2:                    # at most two sample lists in flight
                out, _ = handles.pop(0).result()
                n += len(out[0])
        for h in handles:
            out, _ = h.result()
            n += len(out[0])
        return n, d2h_bytes(out)

    e2e = e2e_pipe = None
    plain_n = pipe_n = 0
    plain_s = pipe_s = 1.0
    d2h_plain = d2h_pipe = 0
    if not args.no_e2e:
        pairs = [make_pair(0), make_pair(1)]
        torch.cuda.synchronize()
        out = None
        for _ in range(max(3, min(args.warmup, 5))):     # (holding the previous batch like the timed loop does, so
            out = plain_batch(pairs[0])                  #  that both generations of page-locked blocks exist)
        rig.barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            out = plain_batch(pairs[0])
            plain_n += len(out[0])
        rig.barrier()
        plain_s = time.perf_counter() - t0
        d2h_plain = d2h_bytes(out)
        del out
        # per-rank timeline of the plain sequence (5 more batches, outside the timed e2e region): where a batch's
        # host wall time goes -- waiting for the rollout, statistics (+ all-reduce) / compaction, the D2H copy
        tl = np.zeros(5)
        smp, pool, _ = pairs[0]
        for _ in range(5):
            ta = time.perf_counter()
            smp.reset(obs_host)
            tb = time.perf_counter()
            while True:
                _, _, _, info = smp.sample(None)
                if info["alive_ratio"] <= 0.1:
                    break
            smp.finish_all_paths()
            tc_ = time.perf_counter()
            dev_out, _ = pool.get_device()
            torch.cuda.synchronize()
            td = time.perf_counter()
            host_out = pool.to_host(dev_out)
            te = time.perf_counter()
            pool.reset()
            tl += np.array([tb - ta, tc_ - tb, td - tc_, te - td, te - ta]) * 1e3 / 5
            del host_out, dev_out
        timeline = torch.tensor(tl, device=dev, dtype=torch.float64)
        if world > 1:
            gathered = [torch.zeros_like(timeline) for _ in range(world)]
            rig.dist.all_gather(gathered, timeline)
        else:
            gathered = [timeline]
        timeline_rows = [[round(float(x), 3) for x in g] for g in gathered]
        pipelined_run(pairs, 4)             # warm-up: page-locked buffer sets of both pairs get allocated
        rig.barrier()
        t0 = time.perf_counter()
        pipe_n, d2h_pipe = pipelined_run(pairs, args.steps)
        rig.barrier()
        pipe_s = time.perf_counter() - t0

    (ms, dyn_launch_ms, gae_launch_ms, plain_s, pipe_s), (n_tr, launches, plain_n, pipe_n) = \
        rig.reduce_result(res, extra_max=(plain_s, pipe_s), extra_sum=(plain_n, pipe_n))
    if rank != 0:
        return
    pk = peaks()
    fdyn, fact, fvvc = rig.flops()
    gae_steps = B * (T - 1)
    gae_gbs = 32.0 * gae_steps / (gae_launch_ms * 1e-3) / 1e9 if gae_launch_ms > 0 else 0.0
    # CPU baseline: rank 0 at N=1 only (under torchrun OMP_NUM_THREADS is pinned to 1)
    skip_cpu = world > 1 or args.cpu_batch <= 0        # --cpu-batch 0: developer runs only
    cpu = None
    if not skip_cpu:
        cpu_n, cpu_dt = cpu_rollout_sample(args.cpu_batch)
        if cpu_dt < 6.0:                                # scale the bounded sample to ~12 s of CPU work
            scaled = int(min(20000, args.cpu_batch * 12.0 / max(cpu_dt, 1e-3)))
            cpu_n, cpu_dt = cpu_rollout_sample(scaled)
            args.cpu_batch = scaled
        rows_s, rows_dt = cpu_single_step(10000)
        trows_s, trows_dt, tthreads = cpu_single_step_torch(10000)
        cpu = {"value": cpu_n / cpu_dt, "unit": UNIT, "cores": host_threads(), "kind": "port",
               "sample": "%d start states x %d steps (one pass, %.1f s)" % (args.cpu_batch, T - 1, cpu_dt),
               "single_step": {"rows_per_s": rows_s, "rows": 10000, "seconds": rows_dt,
                               "what": "BASELINE configs[0] / BASELINE.md B1: one FakeEnv.step (predict_ensemble + KL + "
                                       "statics) on 10k (obs17, act6) rows, oracle port (numpy)"},
               "single_step_torch_bmm": {"rows_per_s": trows_s, "rows": 10000, "seconds": trows_dt, "threads": tthreads,
                                         "what": "BASELINE.md B2: the same step with the ensemble GEMMs through torch-CPU bmm"},
               "gae": cpu_gae_reference_ms_per_1m()}
    line = base_line(rig, args, cfg, n_tr / (ms * 1e-3), ms / args.steps, {
        "start_states_per_gpu": B,
        "l2": "rollout buffers (%.0f MB/GPU) exceed the 126 MB L2; no explicit flush" %
              (B * T * ((2 * rig.O + 2 * rig.A + 11) * 4 + 1) / 1e6),
        "flop_per_transition": fdyn + fact + fvvc})
    line["roofline"] = roofline_obj(pk, fdyn, B, dyn_launch_ms, ms / args.steps, T - 1, "dynamics-ensemble GEMM chain (K1)")
    line["gae"] = {"ms_per_1M_steps": gae_launch_ms / (gae_steps / 1e6), "achieved_GBps": gae_gbs,
                   "peak_GBps": pk["hbm"], "frac": gae_gbs / pk["hbm"], "bytes_per_step": 32,
                   "steps_per_launch": gae_steps, "scan": "strict float64 sequential (bit-exact)"}
    line["cpu_baseline"] = cpu
    if not args.no_e2e:
        line["e2e"] = {"value": plain_n / plain_s, "unit": UNIT, "h2d_bytes_per_step": int(obs_host.nbytes),
                       "d2h_bytes_per_step": int(d2h_plain), "batches": args.steps,
                       "api": "the unmodified caller's sequence (cmbpo.py:251-269): ModelSampler.reset / sample / "
                              "finish_all_paths + blocking ModelBuffer.get(), numpy in, caller-owned numpy out, one pair"}
        d2h_ms = float(np.mean([r[3] for r in timeline_rows]))
        line["e2e_timeline"] = {"columns": ["reset_h2d_ms", "rollout_wait_sample_finish_ms", "stats_allreduce_compact_ms",
                                            "d2h_ms", "total_ms"], "per_rank": timeline_rows,
                                "d2h_GBps_per_rank": d2h_plain / (d2h_ms * 1e-3) / 1e9 if d2h_ms > 0 else None,
                                "d2h_GBps_aggregate": world * d2h_plain / (d2h_ms * 1e-3) / 1e9 if d2h_ms > 0 else None,
                                "numa_local_cores": args.numa_cores,
                                "note": "5 batches of the plain sequence per rank, host wall clock per stage"}
        line["e2e_pipelined"] = {"value": pipe_n / pipe_s, "unit": UNIT, "h2d_bytes_per_step": int(obs_host.nbytes),
                                 "d2h_bytes_per_step": int(d2h_pipe), "batches": args.steps,
                                 "api": "two sampler+buffer pairs alternating with ModelBuffer.get_async().result() "
                                        "(extension: views of recycled page-locked buffers); batch i+1 rolls out while "
                                        "batch i is collected and copied"}
    else:
        line["e2e"] = None
    line["breakdown_ms_per_step"] = {"dynamics_gemm_chain": res["dyn_ms"] / args.steps, "policy_pass": res["pol_ms"] / args.steps,
                                     "row_kernel": res["step_ms"] / args.steps, "gae": res["gae_ms"] / args.steps,
                                     "note": "rank 0, CUDA events around each launch"}
    line["gpu_launches"] = int(launches)
    line["clocks"] = res["clocks"]
    emit(line)


# ---- configs[2]: AntSafe, 1M start states sharded (strong scaling) -----------------------------------
def bench_hcs_unc(rig, args, cfg):
    """The reference's default rollout mode: the limit is calibrated like cmbpo.py:198-200 (depth x mean one-step KL)."""
    obs, act = rig.wl.make_states(7, 5000, rig.O, rig.A, rig.dyn)
    out = rig.eng.fakeenv_step(rig.env_cfg, obs, act, seed=1, step=0)
    rig.unc_mode, rig.dkl_lim = True, 5.0 * float(out["dkl_path"].mean())
    cfg = dict(cfg, total=cfg["total_per_gpu"] * rig.world)
    bench_ant1m(rig, args, cfg)


def bench_ant1m(rig, args, cfg):
    world = rig.world
    total = args.total if args.total > 0 else cfg["total"]
    B, T = total // world, MAXROLL
    res = rig.timed_rollouts(B, T, args.steps, args.warmup)
    (ms, dyn_launch_ms, gae_launch_ms), (n_tr, launches) = rig.reduce_result(res)
    if rig.rank != 0:
        return
    pk = peaks()
    fdyn, fact, fvvc = rig.flops()
    line = base_line(rig, args, cfg, n_tr / (ms * 1e-3), ms / args.steps, {
        "start_states_total": B * world, "start_states_per_gpu": B,
        "mean_path_length": n_tr / args.steps / (B * world),
        "l2": "rollout buffers far exceed the 126 MB L2; no explicit flush",
        "flop_per_transition": fdyn + fact + fvvc})
    # rows per dynamics launch vary (alive-row compaction): the achieved rate uses the FLOPs of the rows that were
    # stored (= useful work) over the summed launch time
    useful = fdyn * (n_tr / world) / (res["dyn_ms"] * 1e-3) / 1e12 if res["dyn_ms"] > 0 else 0.0
    line["roofline"] = {"bound": "tensor", "kernel": "dynamics-ensemble GEMM chain (K1), all launches of the pass",
                        "achieved": useful, "peak": pk["tf_burst"], "unit": "TFLOP/s", "frac": useful / pk["tf_burst"],
                        "frac_burst": useful / pk["tf_burst"], "frac_sustained": useful / pk["tf_sus"], "traffic": None,
                        "note": "useful FLOPs (stored transitions of rank 0) / summed K1 time of rank 0; rows of paths "
                                "that ended since the last compaction are computed and discarded"}
    line["writeout_GBps"] = rig.row_bytes() * n_tr / (ms * 1e-3) / 1e9
    line["cpu_baseline"] = None
    line["e2e"] = None
    line["breakdown_ms_per_step"] = {"dynamics_gemm_chain": res["dyn_ms"] / args.steps, "policy_pass": res["pol_ms"] / args.steps,
                                     "row_kernel": res["step_ms"] / args.steps, "gae": res["gae_ms"] / args.steps}
    line["gpu_launches"] = int(launches)
    line["clocks"] = res["clocks"]
    emit(line)


# ---- configs[3]: HumanoidSafe rollout -> GAE, plus the standalone GAE layouts of SURVEY.md 8d -------------
def gae_layouts(rig):
    """Standalone GAE + cost-GAE timings (CUDA events, 20 launches after 3 warm-ups), ms per 1M steps and GB/s
    at 32 B/step: ModelBuffer layout full / ragged, CPOBuffer flat layout, and the amortised 64M-step launch."""
    torch, eng, L = rig.torch, rig.eng, rig.L
    g = torch.Generator(device=rig.dev)
    g.manual_seed(1)
    out = {}

    def rnd(*shape):
        return torch.randn(*shape, device=rig.dev, generator=g)

    def timeit(fn, n=20):
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    def paths_case(name, B, T, ragged):
        r, v, c, cv = rnd(T, B), rnd(T, B), (torch.rand(T, B, device=rig.dev, generator=g) < 0.1).float(), rnd(T, B)
        length = (torch.randint(1, T, (B,), device=rig.dev, generator=g) if ragged
                  else torch.full((B,), T - 1, device=rig.dev)).to(torch.int32)
        lv, lc = rnd(B), rnd(B)
        outs = tuple(torch.zeros(T, B, device=rig.dev) for _ in range(4))
        steps = int(length.sum().item())
        ms = timeit(lambda: eng.gae_paths(r, v, c, cv, length, lv, lc, GAE["gamma"], GAE["lam"], GAE["cost_gamma"],
                                          GAE["cost_lam"], B, T, 1, B, out=outs))
        out[name] = {"steps": steps, "ms": ms, "ms_per_1M_steps": ms / (steps / 1e6), "GBps": 32.0 * steps / (ms * 1e-3) / 1e9}

    paths_case("modelbuffer_32768x35_full", 32768, 35, False)
    paths_case("modelbuffer_32768x35_ragged", 32768, 35, True)
    paths_case("amortised_64M_steps", 1900000, 35, False)
    # CPOBuffer flat layout: 1049 paths x 1000 steps (warp-shuffle segmented scan)
    n_seg, seg = 1049, 1000
    n = n_seg * seg
    r, v, cv = rnd(n), rnd(n), rnd(n)
    c = (torch.rand(n, device=rig.dev, generator=g) < 0.1).float()
    off = torch.arange(0, n + 1, seg, device=rig.dev, dtype=torch.int64)
    lv, lc = rnd(n_seg), rnd(n_seg)
    outs = tuple(torch.zeros(n, device=rig.dev) for _ in range(4))
    for nm, scan in (("cpobuffer_flat_1049x1000_warp", L.SCAN_WARP), ("cpobuffer_flat_1049x1000_strict", L.SCAN_STRICT)):
        ms = timeit(lambda: eng.gae_flat(r, v, c, cv, off, lv, lc, GAE["gamma"], GAE["lam"], GAE["cost_gamma"],
                                         GAE["cost_lam"], out=outs, scan=scan))
        out[nm] = {"steps": n, "ms": ms, "ms_per_1M_steps": ms / (n / 1e6), "GBps": 32.0 * n / (ms * 1e-3) / 1e9}
    return out


def bench_hs_gae(rig, args, cfg):
    B, T = args.batch, MAXROLL
    res = rig.timed_rollouts(B, T, args.steps, args.warmup)
    (ms, dyn_launch_ms, gae_launch_ms), (n_tr, launches) = rig.reduce_result(res)
    layouts = gae_layouts(rig) if rig.rank == 0 else None
    rig.barrier()
    if rig.rank != 0:
        return
    pk = peaks()
    fdyn, fact, fvvc = rig.flops()
    gae_steps = B * (T - 1)
    gae_gbs = 32.0 * gae_steps / (gae_launch_ms * 1e-3) / 1e9 if gae_launch_ms > 0 else 0.0
    line = base_line(rig, args, cfg, n_tr / (ms * 1e-3), ms / args.steps, {
        "start_states_per_gpu": B, "l2": "rollout buffers exceed the 126 MB L2; no explicit flush",
        "flop_per_transition": fdyn + fact + fvvc})
    line["roofline"] = roofline_obj(pk, fdyn, B, dyn_launch_ms, ms / args.steps, T - 1, "dynamics-ensemble GEMM chain (K1)")
    line["roofline"]["traffic"] = None
    line["roofline"]["tensor_pipe_active_pct_ncu"] = None
    line["gae"] = {"ms_per_1M_steps": gae_launch_ms / (gae_steps / 1e6), "achieved_GBps": gae_gbs, "peak_GBps": pk["hbm"],
                   "frac": gae_gbs / pk["hbm"], "bytes_per_step": 32, "steps_per_launch": gae_steps,
                   "scan": "strict float64 sequential (bit-exact), in the rollout pass"}
    for k in layouts.values():
        k["frac_hbm"] = k["GBps"] / pk["hbm"]
    line["gae_layouts"] = layouts
    line["writeout_GBps"] = rig.row_bytes() * n_tr / (ms * 1e-3) / 1e9
    line["cpu_baseline"] = None
    line["e2e"] = None
    line["breakdown_ms_per_step"] = {"dynamics_gemm_chain": res["dyn_ms"] / args.steps, "policy_pass": res["pol_ms"] / args.steps,
                                     "row_kernel": res["step_ms"] / args.steps, "gae": res["gae_ms"] / args.steps}
    line["gpu_launches"] = int(launches)
    line["clocks"] = res["clocks"]
    emit(line)


# ---- configs[4]: H x B sweep -------------------------------------------------------------------------------
def bench_sweep(rig, args, cfg):
    world = rig.world
    pk = peaks()
    fdyn, fact, fvvc = rig.flops()
    Hs = [int(x) for x in args.sweep_h.split(",")]
    Bs = [int(x) for x in args.sweep_b.split(",")]
    cells, launches_total, clk = [], 0, None
    for Btot in Bs:
        B = max(1, Btot // world)
        for H in Hs:
            steps = max(2, min(args.steps, int(2e8 / max(B * H, 1)) + 2))       # small cells: more repetitions
            last_cell = Btot == Bs[-1] and H == Hs[-1]          # the cell `value` reports is the one dumped
            res = rig.timed_rollouts(B, H + 1, steps, max(1, min(args.warmup, 2)), dump=last_cell)
            (ms, dyn_launch_ms, gae_launch_ms), (n_tr, launches) = rig.reduce_result(res)
            launches_total += launches
            clk = res["clocks"]
            tr_s = n_tr / (ms * 1e-3)
            k1 = fdyn * B / (dyn_launch_ms * 1e-3) / 1e12 if dyn_launch_ms > 0 else 0.0
            cells.append({"H": H, "B_total": B * world, "B_per_gpu": B, "passes": steps, "transitions_per_s": tr_s,
                          "ms_per_pass": ms / steps, "k1_launch_ms": dyn_launch_ms, "k1_TFLOPs": k1,
                          "k1_frac_burst": k1 / pk["tf_burst"], "job_TFLOPs": (fdyn + fact + fvvc) * tr_s / 1e12,
                          "job_frac_burst": (fdyn + fact + fvvc) * tr_s / 1e12 / (pk["tf_burst"] * world),
                          "writeout_GBps": rig.row_bytes() * tr_s / 1e9,
                          "gae_GBps": 32.0 * B * H / (gae_launch_ms * 1e-3) / 1e9 if gae_launch_ms > 0 else None})
            rig.torch.cuda.empty_cache()
    if rig.rank != 0:
        return
    best = max(cells, key=lambda c: c["transitions_per_s"])
    big = cells[-1]
    line = base_line(rig, args, cfg, big["transitions_per_s"], big["ms_per_pass"], {
        "value_is": "the largest cell (H=%d, B_total=%d)" % (big["H"], big["B_total"]), "horizons": Hs, "batches_total": Bs,
        "passes_per_cell": "max(2, min(--steps, 2e8 / (B_per_gpu x H) + 2)), listed as cells[].passes",
        "l2": "cells below ~50k start states per GPU fit the 126 MB L2; no explicit flush",
        "flop_per_transition": fdyn + fact + fvvc})
    line["roofline"] = {"bound": "tensor", "kernel": "dynamics-ensemble GEMM chain (K1), largest cell", "achieved": big["k1_TFLOPs"],
                        "peak": pk["tf_burst"], "unit": "TFLOP/s", "frac": big["k1_frac_burst"], "frac_burst": big["k1_frac_burst"],
                        "frac_sustained": big["k1_TFLOPs"] / pk["tf_sus"], "traffic": None}
    line["cells"] = cells
    line["best_cell"] = best
    line["cpu_baseline"] = None
    line["e2e"] = None
    line["gpu_launches"] = int(launches_total)
    line["clocks"] = clk
    emit(line)


L_PROF_DYN, L_PROF_GAE = 0, 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed passes of the hot path; --config sweep: per cell max(2, min(STEPS, 2e8 / (B x H) + 2)), "
                         "reported as cells[].passes")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--precision", default="fp16", choices=["fp32", "fp16", "bf16"])
    ap.add_argument("--batch", type=int, default=100000, help="start states per GPU")
    ap.add_argument("--cpu-batch", type=int, default=500, help="start states of the bounded CPU sample")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs only: skip the end-to-end legs (e2e = null)")
    ap.add_argument("--config", default="hcs", choices=sorted(CONFIGS), help="BASELINE.json configs[1..4]; default configs[1]")
    ap.add_argument("--mode", default="mean", choices=["mean", "injected"],
                    help="transition mode: deterministic mean (reference behaviour) or mean + std*eps")
    ap.add_argument("--fuse", action="store_true", help="use the fused rollout step (CMBPO_ROLLOUT_FUSE)")
    ap.add_argument("--total", type=int, default=0, help="ant1m: total start states (default 1,000,000)")
    ap.add_argument("--no-numa-bind", action="store_true", help="N > 1: do not pin ranks to their GPU's NUMA-local cores")
    ap.add_argument("--sweep-h", default="1,2,5,10,20,30")
    ap.add_argument("--sweep-b", default="10000,100000,1000000,4000000")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (rank 0; a fixed "
                         "sample of paths, < 64 MB; --config sweep: the last cell, the one `value` reports); the inputs "
                         "depend only on the arguments, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl cuda)")
    # stdout carries exactly ONE JSON line: anything libraries print at C level while the job runs
    # (NCCL's version banner) goes to stderr; the real stdout is restored for the final print
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 1000)] + sys.argv
        os.execv(sys.executable, cmd)
    run_cuda(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
