"""TEST / BENCH INFRASTRUCTURE: build and call ``oracle/cxx_loop.cpp`` - the host (g++ -O3 -fopenmp) build of the
solver sources in ``mpc-code_b200/csrc`` running the closed loop for B instances on all host cores.

This is the CPU arm of ``bench.py`` ("same algorithm, C++"): a baseline, not a checker (it shares its arithmetic with
the device code).  Nothing in the product package imports it.
"""
from __future__ import annotations

import ctypes
import hashlib
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "mpc-code_b200", "csrc")
BUILD = os.path.join(HERE, "_build")
VP = ctypes.c_void_p


def build(name, prob, ss, ocp):
    """Compile the loop for one problem; returns the path of the shared object (cached by content hash)."""
    from mpc_code_b200.build import build_dir_for
    from mpc_code_b200.devicegen import generate_header
    text = generate_header(prob, ss, ocp)["text"]
    hsh = hashlib.sha256(text.encode())
    for fn in ("mpcb_device.cuh", "mpcb_ocp.cuh", "mpcb_target.cuh"):
        with open(os.path.join(CSRC, fn), "rb") as fh:
            hsh.update(fh.read())
    with open(os.path.join(HERE, "cxx_loop.cpp"), "rb") as fh:
        hsh.update(fh.read())
    hsh.update(_cpu_flags().encode())        # -march=native: a library built on another host CPU must not be reused
    digest = hsh.hexdigest()[:16]
    base = build_dir_for(BUILD, "cxx_%s_%s.so" % (name, digest))
    work = os.path.join(base, "cxx_%s_%s" % (name, digest))
    so = os.path.join(base, "cxx_%s_%s.so" % (name, digest))
    if not os.path.exists(so):
        os.makedirs(work, exist_ok=True)
        hdr = os.path.join(work, "mpcb_model.h")
        tmp_h = hdr + ".tmp%d" % os.getpid()
        with open(tmp_h, "w") as fh:
            fh.write(text)
        os.replace(tmp_h, hdr)
        tmp = so + ".tmp%d" % os.getpid()
        subprocess.run(["g++", "-O3", "-march=native", "-fopenmp", "-shared", "-fPIC", "-std=c++17", "-Wno-unknown-pragmas",
                        "-I", work, "-I", CSRC, "-o", tmp, os.path.join(HERE, "cxx_loop.cpp")], check=True)
        os.replace(tmp, so)
    return so


def _cpu_flags() -> str:
    try:
        with open("/proc/cpuinfo") as fh:
            for line in fh:
                if line.startswith("flags"):
                    return line
    except OSError:
        pass
    return ""


class CxxLoop:
    def __init__(self, name, prob, ss, ocp, range_bounds):
        """``range_bounds``: (lbg, ubg) of the range rows stage by stage (as `mpcb_set_const("ocp_lbg")` takes them)."""
        self.prob, self.ss, self.ocp = prob, ss, ocp
        self.lib = ctypes.CDLL(build(name, prob, ss, ocp))
        self.lib.cxx_closed_loop.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_double] + [VP] * 13 + [ctypes.c_int] + \
            [VP] * 5 + [ctypes.c_int] * 3 + [VP] * 3 + [ctypes.c_int, VP]
        self.lbg, self.ubg = [np.ascontiguousarray(v if v.size else np.zeros(1), dtype=float) for v in range_bounds]
        # every core this process may run on, whatever OMP_NUM_THREADS says (torchrun sets it to 1 for its workers)
        try:
            ncpu = len(os.sched_getaffinity(0))
        except AttributeError:
            ncpu = os.cpu_count() or 1
        self.lib.cxx_set_threads.argtypes = [ctypes.c_int]
        self.lib.cxx_set_threads(int(os.environ.get("MPCB_CPU_THREADS", ncpu)))

    def threads(self):
        return int(self.lib.cxx_threads())

    def run(self, nsim, x0_p, x0_m, noise=None, nwarm=0):
        p = self.prob
        x0_p = np.ascontiguousarray(np.atleast_2d(x0_p), dtype=float).copy()
        x0_m = np.ascontiguousarray(np.atleast_2d(x0_m), dtype=float)
        B = x0_p.shape[0]
        sp = np.zeros((nsim, p.nu + p.ny + p.nx))
        for k in range(nsim):
            if p.defSP is not None:
                ysp, usp, xsp = [np.asarray(v, dtype=float).ravel() for v in p.defSP(k * p.h)]
                sp[k] = np.concatenate([usp, ysp, xsp])
        est = p.estimator
        est_type = 0 if est["type"] == "kalss" else 1
        c = lambda a: np.ascontiguousarray(a, dtype=float)  # noqa: E731
        Q = c(est.get("Q", np.zeros((p.nxi, p.nxi)))); R = c(est.get("R", np.zeros((p.ny, p.ny))))
        K = c(est.get("K", np.zeros((p.nxi, p.ny)))).reshape(-1)
        has_db = est["dmin"] is not None
        dmin = c(est["dmin"]) if has_db else np.zeros(max(p.nd, 1)); dmax = c(est["dmax"]) if has_db else np.zeros(max(p.nd, 1))
        P0 = c(est["P0"]).reshape(-1)
        U = np.zeros((nsim, B, p.nu)); it = np.zeros((nsim, B), dtype=np.int32); st = np.zeros((nsim, B), dtype=np.int32)
        timed = np.zeros(B)
        nz = None if noise is None else c(noise)
        ptr = lambda a: a.ctypes.data_as(VP) if a is not None else None  # noqa: E731
        keep = [c(p.u0), c(p.dhat0 if p.nd else np.zeros(1)), c(self.ocp.w_lb), c(self.ocp.w_ub), c(self.ss.w_lb), c(self.ss.w_ub)]
        nth = self.lib.cxx_closed_loop(B, nsim, float(p.h), ptr(x0_p), ptr(x0_m), ptr(keep[0]), ptr(keep[1]), ptr(P0), ptr(nz),
                                       ptr(sp), ptr(keep[2]), ptr(keep[3]), ptr(self.lbg), ptr(self.ubg), ptr(keep[4]),
                                       ptr(keep[5]), est_type, ptr(Q), ptr(R), ptr(K), ptr(dmin), ptr(dmax), 1 if has_db else 0,
                                       int(p.sol_optss["ipopt.max_iter"]), int(p.sol_optdyn["ipopt.max_iter"]),
                                       ptr(U), ptr(it), ptr(st), int(nwarm), ptr(timed))
        return dict(U=U, ITER_DYN=it, STATUS_DYN=st, Xp=x0_p, threads=nth, timed_s=timed)

    def throughput(self, x0, noise, nwarm):
        """Closed-loop instance-steps per second over all threads for the steps after each instance's first `nwarm`
        (cold-start) steps: timed steps / (sum of the per-instance timed seconds / threads)."""
        nsim = noise.shape[0]
        r = self.run(nsim, x0, x0, noise, nwarm=nwarm)
        busy = float(r["timed_s"].sum()) / max(r["threads"], 1)
        return x0.shape[0] * (nsim - nwarm) / busy, r


def range_bounds_of(ocp):
    """Range rows of g_lb/g_ub stage by stage: [Y_k, DU_k, G_k] bounds for k = 0..N-1 (see include/mpcb.h)."""
    o = ocp
    n_dyn = o.n * (o.N + 1) + (o.n if o.term_eq is not None else 0)
    ny_rows = 0 if o.yFree else o.p * o.N
    ndu_rows = 0 if o.DuFree else o.m * o.N
    ngin_rows = o.n_gin * o.N

    def per_stage(v):
        blocks = []
        if ny_rows:
            blocks.append(v[n_dyn:n_dyn + ny_rows].reshape(o.N, o.p))
        if ndu_rows:
            blocks.append(v[n_dyn + ny_rows:n_dyn + ny_rows + ndu_rows].reshape(o.N, o.m))
        if ngin_rows:
            o3 = n_dyn + ny_rows + ndu_rows
            blocks.append(v[o3:o3 + ngin_rows].reshape(o.N, o.n_gin))
        return np.ascontiguousarray(np.hstack(blocks).reshape(-1)) if blocks else np.zeros(0)
    return per_stage(o.g_lb), per_stage(o.g_ub)
