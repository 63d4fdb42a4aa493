"""Rollout throughput of a deep dynamics model: HumanoidSafe (obs 47, act 17) with the reference's code-default
dynamics architecture (200, 200, 200, 200) (algorithms/cmbpo.py:54), a probabilistic 96-output ensemble of 7.
Device-resident rollout + GAE over B start states, deterministic-mean transitions, at each precision; prints the card
and its power limit with the numbers.
usage: python tools/deep_rollout_rate.py [B] [maxroll] [precisions, comma separated]"""
import os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import cmbpo_b200 as cb
from cmbpo_b200 import _lib as L
from cmbpo_b200 import workload as wl

B = int(sys.argv[1]) if len(sys.argv) > 1 else 100000
T = int(sys.argv[2]) if len(sys.argv) > 2 else 35
PRECS = sys.argv[3].split(",") if len(sys.argv) > 3 else ["fp16", "fp32"]
O, A, HIDDEN = 47, 17, (200, 200, 200, 200)

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
print("card: %s" % card)
dyn, actor, v, vc = wl.make_problem(0, O, A, hidden=HIDDEN, task="HumanoidSafe-v2")
eng = cb.Engine(0, precision="fp32")
cb.B200PE.from_arrays(eng, L.NET_DYN, dyn)
pol = cb.B200Policy(eng)
pol.load_actor(actor.W, actor.b, actor.log_std)
pol.load_values(v, vc)
obs, _ = wl.make_states(1, B, O, A, dyn)
cfg = L.EnvCfg(L.TERM_NO_DONE, L.COST_ZERO, 0, 1, 1)
bufs = cb.RolloutBuffers(eng, B, T, O, A)
bufs.set_inputs(obs)
for prec in PRECS:
    for i in range(2):
        bufs.run(cfg, seed=i, precision=prec)
        bufs.gae(0.99, 0.95, 0.97, 0.5)
    torch.cuda.synchronize()
    reps = 5
    t0 = time.perf_counter()
    n = 0
    for i in range(reps):
        bufs.run(cfg, seed=10 + i, precision=prec)
        bufs.gae(0.99, 0.95, 0.97, 0.5)
        n += int(bufs.length.sum().item())
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / reps
    print("%s: dynamics %s -> %d outputs, B = %d, maxroll %d: %.2f ms per rollout, %.2f M transitions/s"
          % (prec, "x".join(map(str, HIDDEN)), dyn.W[-1].shape[-1], B, T, dt * 1e3, n / reps / dt / 1e6))
eng.close()
