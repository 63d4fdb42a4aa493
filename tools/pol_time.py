"""A/B aid: host-clock time of the policy pass (the grouped tcgen05 kernel of the merged actor + V + VC ensemble).
usage: [CMBPO_B200_LIB=tools/lib_x.so] python tools/pol_time.py [rows]"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import cmbpo_b200 as cb
from cmbpo_b200 import workload as orc

N = int(sys.argv[1]) if len(sys.argv) > 1 else 100000
dyn, actor, v, vc = orc.make_problem(0, 17, 6, hidden=(64, 64))
eng = cb.Engine(0, precision="fp16")
pol = cb.B200Policy(eng)
pol.load_actor(actor.W, actor.b, actor.log_std)
pol.load_values(v, vc)
obs, act = orc.make_states(1, N, 17, 6, dyn)
x = eng.to_device(obs)
for i in range(3):
    eng.policy_act(x)
torch.cuda.synchronize()
t0 = time.perf_counter()
for i in range(5):
    eng.policy_act(x)
torch.cuda.synchronize()
print("policy_act %d rows: %.3f ms" % (N, (time.perf_counter() - t0) / 5 * 1e3))
