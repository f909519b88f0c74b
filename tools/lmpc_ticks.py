import os, sys, time; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import __graft_entry__ as entry
from mpc_code_b200.mpc_loop import CompiledProblem
prob, ss, ocp = entry._problem("lmpc_cstr")
B = 4096
ctl = CompiledProblem(prob, "lmpc_cstr").controller(B)
ctl.reset(); ctl.h.set_groups(1)
rows = []
for k in range(100):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); o = ctl.step_fused(); e1.record(); torch.cuda.synchronize()
    rows.append((k, e0.elapsed_time(e1), ctl.h.last_ticks, int((o["STATUS_DYN"] == 2).sum()), float(o["ITER_DYN"].float().mean())))
ms = np.array([r[1] for r in rows])
print("mean ms %.2f median %.2f" % (ms.mean(), np.median(ms)))
for r in rows:
    if r[3] > 0 or r[1] > 1.5 * np.median(ms) or r[0] < 3:
        print("step %d: %.2f ms, ticks %d, infeasible %d, mean iters %.1f" % r)
