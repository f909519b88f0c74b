import os, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from mpc_code_b200.mpc_loop import CompiledProblem
prob, ss, ocp = bench._problem()
B, K = bench.BATCH_PER_GPU, 20
cp = CompiledProblem(prob, "nmpc_cstr")
x0, noise = bench._workload(prob, B, K + 5)
ctl = cp.controller(B); ctl.reset(x0_p=x0, x0_m=x0); ctl.h.set_groups(int(os.environ.get("G", "1")))
nz = torch.as_tensor(noise, device=ctl.h.device)
for k in range(5): ctl.step_fused(nz[k])
torch.cuda.synchronize()
h = ctl.h
import types
acc = {}
def wrap(obj, name):
    f = getattr(obj, name)
    def g(*a, **kw):
        t0 = time.perf_counter(); r = f(*a, **kw); acc.setdefault(name, []).append(time.perf_counter() - t0); return r
    setattr(obj, name, g)
for n in ("plant_meas", "step", "plant_step"):
    wrap(h, n)
wrap(ctl, "_params"); wrap(ctl, "_row")
for k in range(5, 5 + K):
    ctl.step_fused(nz[k])
torch.cuda.synchronize()
for n, v in acc.items():
    print("%-12s calls %3d median %.0f us  max %.0f us" % (n, len(v), 1e6 * np.median(v), 1e6 * max(v)))
