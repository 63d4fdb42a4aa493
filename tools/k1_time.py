"""A/B aid: CUDA-event time of the dynamics GEMM chain (K1) alone, via the library's own profiling slots.
usage: [CMBPO_B200_LIB=tools/lib_x.so] python tools/k1_time.py [rows] [hidden] [obs] [act] [layers] [precision]
layers = number of hidden layers of width `hidden` (default 2); precision = fp16 (default), bf16 or fp32.  The
dynamics net has 2 (obs + 1) outputs: HumanoidSafe (obs 47, act 17) with 4 layers of 200 is a 96-output deep net."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import cmbpo_b200 as cb
from cmbpo_b200 import _lib as L
from cmbpo_b200 import workload as orc

N = int(sys.argv[1]) if len(sys.argv) > 1 else 100000
H = int(sys.argv[2]) if len(sys.argv) > 2 else 512
O = int(sys.argv[3]) if len(sys.argv) > 3 else 17
A = int(sys.argv[4]) if len(sys.argv) > 4 else 6
NH = int(sys.argv[5]) if len(sys.argv) > 5 else 2
PREC = sys.argv[6] if len(sys.argv) > 6 else "fp16"
dyn, actor, v, vc = orc.make_problem(0, O, A, hidden=(H,) * NH)
if os.environ.get("K1_ZERO"):      # data-dependence probe: all-zero weights and biases (same instruction stream)
    for w in dyn.W: w[...] = 0
    for b in dyn.b: b[...] = 0
eng = cb.Engine(0, precision=PREC)
model = cb.B200PE.from_arrays(eng, L.NET_DYN, dyn)
obs, act = orc.make_states(1, N, O, A, dyn)
x = eng.to_device(np.concatenate([obs, act], -1))
for i in range(5):
    model.predict_ensemble_device(x)
torch.cuda.synchronize()
eng.profile(True)
eng.profile_read(0, True)
for i in range(40):
    model.predict_ensemble_device(x)
torch.cuda.synchronize()
ms, n = eng.profile_read(0, True)
print("%s K1 %d rows H=%d x %d layers, %d outputs, %s: %.4f ms per launch (%d launches)"
      % (os.environ.get("CMBPO_B200_LIB", "default"), N, H, NH, dyn.W[-1].shape[-1], PREC, ms / max(n, 1), n))
