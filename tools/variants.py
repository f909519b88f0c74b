#!/usr/bin/env python
"""Build (here) and time (on the GPU box) several nvcc-flag variants of the problem library with bench.py.

    python tools/variants.py build            # compiles every variant into mpc-code_b200/_build/
    python tools/variants.py run [steps]      # runs bench.py per variant, prints value + kernel time shares
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VARIANTS = {
    "default": "",
    "full_first_eval": "-DMPCB_EVAL_FIRST=0",
}
# KKT kernel occupancy (profiles/r02_variants_kktocc.txt): "-DMPCB_KKT_MINBLOCKS=1" (118 regs) | "=5" (96) | "=6" (80)
# round-2 register/occupancy sweep of k_ocp_eval (profiles/r02_variants_*.txt):
#   "" (128x3, 168 regs) | -DMPCB_EVAL_MINBLOCKS=2 (254 regs, the default since) |
#   -DMPCB_EVAL_BLOCK=64 -DMPCB_EVAL_MINBLOCKS=5 -DMPCB_EVAL_MAXNREG=200 | -DMPCB_EVAL_BLOCK=32 -DMPCB_EVAL_MINBLOCKS=9 -DMPCB_EVAL_MAXNREG=224

if __name__ == "__main__":
    mode = sys.argv[1]
    for name, flags in VARIANTS.items():
        env = dict(os.environ, MPCB_EXTRA_FLAGS=flags)
        if mode == "build":
            subprocess.run([sys.executable, "-c", "import sys; sys.path.insert(0, %r); import __graft_entry__ as e; "
                            "from mpc_code_b200.build import build_library; p, s, o = e._problem(); "
                            "print(%r, build_library('nmpc_cstr', p, s, o)['so'])" % (ROOT, name)], env=env, check=True)
        else:
            steps = sys.argv[2] if len(sys.argv) > 2 else "10"
            res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", steps, "--warmup", "4", "--no-cpu-baseline"],
                                 env=env, capture_output=True, text=True)
            try:
                d = json.loads(res.stdout.strip().splitlines()[-1])
                sh = d["roofline"]["kernel_time_share"]
                print("%-24s value %9.0f e2e %9.0f ms/step %6.2f eval_ms %7.1f  shares: %s" % (
                    name, d["value"], d["e2e"]["value"], d["ms_per_step"], d["roofline"]["kernel_ms_total"],
                    " ".join("%s=%.2f" % (k.replace("ocp_", ""), v) for k, v in sh.items() if v > 0.01)), flush=True)
            except Exception as exc:
                print(name, "FAILED", exc, res.stderr[-400:])
