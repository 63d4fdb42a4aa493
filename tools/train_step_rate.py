"""Device time of one ensemble training step (cmbpo_ens_train_step) in fp32, TF32 and bf16, against an eager-torch
bf16 step (torch.bmm + autograd + torch.optim.Adam: library bf16 GEMMs without fusion), and the wall time of one
B200PE.train call.  Prints the card and its power limit with the numbers.

Per-step time: CUDA events around `STEPS` back-to-back steps on one pre-gathered batch after `WARM` warm-up steps
(a launch-bound step shows the host's enqueue rate here), and the kernels' own time per step from torch.profiler
(the device-busy time).  train(): 50 k rows, batch 256, 5 epochs, no holdout; compared with steps x the event time
per step, the rest is the host loop (two gathers and a ctypes call per step).
usage: python tools/train_step_rate.py [steps] [warm-up]"""
import json, os, subprocess, sys, tempfile, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import cmbpo_b200 as cb
from cmbpo_b200 import _lib as L
from cmbpo_b200 import workload as wl

STEPS = int(sys.argv[1]) if len(sys.argv) > 1 else 300
WARM = int(sys.argv[2]) if len(sys.argv) > 2 else 30
BS = 256
# name: obs, act, hidden, probabilistic, members
SHAPES = {"HCS dynamics 7x(512,512)": (17, 6, (512, 512), True, 7),
          "HumanoidSafe dynamics 7x(200,200,200,200)": (47, 17, (200, 200, 200, 200), True, 7),
          "V 3x(128,128)": (17, 6, (128, 128), False, 3)}

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
print("card: %s" % card)
eng = cb.Engine(0, precision="fp32")


def problem(O, A, hidden, prob, E):
    dyn, _, v, _ = wl.make_problem(0, O, A, hidden=hidden, num_nets=E, vf_nets=E, vf_hidden=hidden)
    ens = dyn if prob else v
    which = L.NET_DYN if prob else L.NET_V
    Din, D = (O + A, O + 1) if prob else (O, 1)
    rng = np.random.default_rng(1)
    x = torch.tensor(rng.standard_normal((E, BS, Din)), dtype=torch.float32, device="cuda")
    y = torch.tensor(rng.standard_normal((E, BS, D)) * 0.1, dtype=torch.float32, device="cuda")
    return ens, which, x, y


def timed(fn, label=None):
    for _ in range(WARM):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(STEPS):
        fn()
    b.record()
    torch.cuda.synchronize()
    event_ms = a.elapsed_time(b) / STEPS
    n = 50
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        prof.export_chrome_trace(os.path.join(d, "t.json"))
        with open(os.path.join(d, "t.json")) as f:
            ev = json.load(f)["traceEvents"]
    kern = [e for e in ev if e.get("cat") in ("kernel", "gpu_memset", "gpu_memcpy")]
    if label:                                      # where the device time of one step goes, by kernel
        per = {}
        for e in kern:
            k = e["name"].replace("(anonymous namespace)::", "").replace("void ", "").split("(")[0][-40:]
            per[k] = per.get(k, 0.0) + e.get("dur", 0) / n
        print("    %s kernels, us per step: %s" % (label, ", ".join("%s %.1f" % kv for kv in sorted(per.items(), key=lambda kv: -kv[1]))))
    return event_ms, sum(e.get("dur", 0) for e in kern) / n / 1000.0


def eager_step(ens, x, y, prob, decay=1e-4):
    """The same step in eager torch: bf16 operands for the GEMMs, fp32 elsewhere; TF's decays (pe_factory.py)."""
    Ws = [torch.tensor(w, device="cuda", requires_grad=True) for w in ens.W]
    bs_ = [torch.tensor(b.reshape(b.shape[0], 1, -1), device="cuda", requires_grad=True) for b in ens.b]
    mu = torch.tensor(ens.mu_in, device="cuda")
    sig = torch.tensor(np.maximum(np.sqrt(ens.var_in), 1e-2), device="cuda")
    opt = torch.optim.Adam(Ws + bs_, lr=1e-3, eps=1e-8)
    nl = len(Ws)
    wd = [decay / 4 if l == 0 else (decay if l == nl - 1 else decay / 2) for l in range(nl)]
    D = y.shape[-1]

    def step():
        a = (x - mu) / sig
        for l in range(nl):
            z = torch.bmm(a.bfloat16(), Ws[l].bfloat16()).float() + bs_[l]
            a = torch.nn.functional.silu(z) if l + 1 < nl else z
        if prob:
            mean, logvar = a[..., :D], a[..., D:]
            s = (mean - y) ** 2
            q = (logvar.exp() - s.detach()) ** 2
            ratio = (0.05 * s.mean() / q.mean()).detach()
            total = (s.mean(dim=(1, 2)) + (ratio * q).mean(dim=(1, 2))).sum() + len(Ws[0]) * 0.05 * (logvar ** 2).mean()
        else:
            total = (0.5 * (a - y) ** 2).mean(dim=(1, 2)).sum()
        total = total + sum(w_ * 0.5 * (W_ ** 2).sum() for w_, W_ in zip(wd, Ws))
        opt.zero_grad(set_to_none=True)
        total.backward()
        opt.step()
    return step


print("per Adam step at bs = %d (%d steps after %d warm-up; ms per step: events / kernels only)" % (BS, STEPS, WARM))
for name, (O, A, hidden, prob, E) in SHAPES.items():
    ens, which, x, y = problem(O, A, hidden, prob, E)
    row = []
    for math in ("fp32", "tf32", "bf16"):
        model = cb.B200PE.from_arrays(eng, which, ens)
        model.configure_training(math=math)
        eng.train_begin(which)
        n0 = eng.launch_count
        eng.train_step(which, x, y, model._train_cfg)
        eng.train_step(which, x, y, model._train_cfg)
        launches = eng.launch_count - n0
        ev, kern = timed(lambda: eng.train_step(which, x, y, model._train_cfg), "%s %s" % (name.split()[0], math))
        row.append("%s %.4f / %.4f (%d launches / 2 steps)" % (math, ev, kern, launches))
    ev, kern = timed(eager_step(ens, x, y, prob))
    row.append("eager-torch bf16 %.4f / %.4f" % (ev, kern))
    print("  %s: %s" % (name, "; ".join(row)))

print("B200PE.train, HCS dynamics, 50 k rows, batch 256, 5 epochs, no holdout")
O, A = 17, 6
rng = np.random.RandomState(0)
n = 50000
X = rng.standard_normal((n, O + A)).astype(np.float32)
M = (rng.standard_normal((O + A, O + 1)) * 0.3).astype(np.float32)
Y = (np.tanh(X @ M) + 0.05 * rng.standard_normal((n, O + 1))).astype(np.float32)
ens, which, x, y = problem(O, A, (512, 512), True, 7)
for math in ("fp32", "tf32", "bf16", "fp32", "tf32", "bf16"):
    model = cb.B200PE.from_arrays(eng, which, ens)
    model.configure_training(math=math, use_scaler_in=True, use_scaler_out=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    model.train(X, Y, batch_size=256, max_epochs=5, holdout_ratio=0.0, rng=np.random.RandomState(1))
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    print("  %s: %.3f s for %d steps (%.4f ms per step)" % (math, wall, model._grad_updates, 1e3 * wall / model._grad_updates))
