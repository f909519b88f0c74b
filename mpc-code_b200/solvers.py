"""ctypes binding of the per-problem CUDA library and CasADi-style batched solver objects.

The reference's loop talks to its solvers as ``sol = solver(lbx=, ubx=, x0=, p=, lbg=, ubg=)`` then
``sol["x"]``, ``sol["f"]`` and ``solver.stats()['return_status']`` (``MPC_code.py:704-718,776-788``).
`BatchedNlpSolver` keeps that convention for a whole batch: ``x0`` is ``[B, nw]``, ``p`` is
``[B, npar]`` (torch CUDA float64 tensors, or anything convertible), and ``stats()`` returns one
status per instance.  All arithmetic happens in the CUDA library; if it cannot be built or loaded
the constructor raises - there is no CPU fallback.
"""
from __future__ import annotations

import ctypes
from typing import Dict, Optional

import numpy as np

STATUS_NAMES = {0: "Solve_Succeeded", 1: "Solved_To_Acceptable_Level", 2: "Infeasible_Problem_Detected",
                -1: "Maximum_Iterations_Exceeded", -2: "Restoration_Failed", -3: "Error_In_Step_Computation",
                -13: "Invalid_Number_Detected"}


class MpcbDims(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int) for n in (
        "nx", "nu", "ny", "nd", "npx", "npy", "nxp", "npxp", "npyp", "nxi", "N", "Mx", "nw", "npar", "ng",
        "nwss", "nparss", "has_ocp", "has_target")]


class MpcbOpts(ctypes.Structure):
    _fields_ = [("max_iter", ctypes.c_int), ("tol", ctypes.c_double), ("mu_init", ctypes.c_double),
                ("bound_relax_factor", ctypes.c_double), ("honor_original_bounds", ctypes.c_int),
                ("bound_push", ctypes.c_double), ("acceptable_tol", ctypes.c_double), ("acceptable_iter", ctypes.c_int)]


C_SYMBOLS = ("mpcb_abi_version", "mpcb_default_opts", "mpcb_get_dims", "mpcb_model_flops", "mpcb_create",
             "mpcb_destroy", "mpcb_last_error", "mpcb_set_const", "mpcb_estimate", "mpcb_target", "mpcb_ocp",
             "mpcb_plant_meas", "mpcb_plant_step", "mpcb_model_output", "mpcb_model_step", "mpcb_stage_derivs",
             "mpcb_last_launches", "mpcb_last_ticks", "mpcb_total_launches", "mpcb_set_groups", "mpcb_set_policy", "mpcb_set_profiling", "mpcb_get_profile", "mpcb_dfma_peak",
             "mpcb_loop_reset", "mpcb_step", "mpcb_loop_get",
             "mpcb_ocp_sens_size", "mpcb_ocp_sens_factor", "mpcb_ocp_jvp", "mpcb_ocp_vjp",
             "mpcb_ocp_sens_size_p", "mpcb_ocp_sens_factor_p", "mpcb_ocp_jvp_p", "mpcb_ocp_vjp_p",
             "mpcb_target_sens_size", "mpcb_target_sens_factor", "mpcb_target_jvp", "mpcb_target_vjp")


class MpcbLibrary:
    """The C ABI of ``include/mpcb.h`` loaded from one compiled problem library."""

    def __init__(self, so_path: str):
        self.path = so_path
        self.lib = ctypes.CDLL(so_path)
        L, vp, ci = self.lib, ctypes.c_void_p, ctypes.c_int
        for name in C_SYMBOLS:
            if not hasattr(L, name):
                raise RuntimeError("%s does not export %s" % (so_path, name))
        L.mpcb_abi_version.restype = ci
        L.mpcb_default_opts.argtypes = [ctypes.POINTER(MpcbOpts)]
        L.mpcb_get_dims.argtypes = [ctypes.POINTER(MpcbDims)]
        L.mpcb_model_flops.argtypes = [ctypes.c_char_p]; L.mpcb_model_flops.restype = ctypes.c_long
        L.mpcb_create.argtypes = [ci, ctypes.POINTER(MpcbOpts), ctypes.POINTER(MpcbOpts), ctypes.POINTER(vp)]
        L.mpcb_destroy.argtypes = [vp]
        L.mpcb_last_error.argtypes = [vp]; L.mpcb_last_error.restype = ctypes.c_char_p
        L.mpcb_set_const.argtypes = [vp, ctypes.c_char_p, vp, ci]
        L.mpcb_estimate.argtypes = [vp, ci] + [vp] * 8
        L.mpcb_target.argtypes = [vp] * 7
        L.mpcb_ocp.argtypes = [vp] * 7
        L.mpcb_plant_meas.argtypes = [vp] * 9
        L.mpcb_plant_step.argtypes = [vp] * 7
        L.mpcb_model_output.argtypes = [vp] * 8
        L.mpcb_model_step.argtypes = [vp] * 8
        L.mpcb_stage_derivs.argtypes = [vp] * 9
        L.mpcb_last_launches.argtypes = [vp]; L.mpcb_last_ticks.argtypes = [vp]
        L.mpcb_total_launches.argtypes = [vp]; L.mpcb_total_launches.restype = ctypes.c_long
        L.mpcb_set_groups.argtypes = [vp, ctypes.c_int]
        L.mpcb_set_policy.argtypes = [vp, ctypes.c_int]
        L.mpcb_set_profiling.argtypes = [vp, ci]
        L.mpcb_get_profile.argtypes = [vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_long),
                                       ctypes.POINTER(ctypes.c_ulonglong)]
        L.mpcb_dfma_peak.argtypes = [ci, ctypes.POINTER(ctypes.c_double)]
        L.mpcb_loop_reset.argtypes = [vp] * 5
        L.mpcb_step.argtypes = [vp, ci] + [vp] * 15
        L.mpcb_loop_get.argtypes = [vp] * 5
        L.mpcb_ocp_sens_size.restype = ctypes.c_long
        L.mpcb_ocp_sens_factor.argtypes = [vp] * 5
        L.mpcb_ocp_jvp.argtypes = [vp, vp, ci, vp, vp, vp]
        L.mpcb_ocp_vjp.argtypes = [vp] * 5
        L.mpcb_ocp_sens_size_p.restype = ctypes.c_long
        L.mpcb_ocp_sens_factor_p.argtypes = [vp] * 5
        L.mpcb_ocp_jvp_p.argtypes = [vp, vp, ci, vp, vp, vp]
        L.mpcb_ocp_vjp_p.argtypes = [vp] * 5
        L.mpcb_target_sens_size.restype = ctypes.c_long
        L.mpcb_target_sens_factor.argtypes = [vp] * 6
        L.mpcb_target_jvp.argtypes = [vp, vp, ci, vp, vp, vp]
        L.mpcb_target_vjp.argtypes = [vp] * 5
        self.dims = MpcbDims()
        L.mpcb_get_dims(ctypes.byref(self.dims))

    def default_opts(self) -> MpcbOpts:
        o = MpcbOpts()
        self.lib.mpcb_default_opts(ctypes.byref(o))
        return o

    def model_flops(self, name: str) -> int:
        return int(self.lib.mpcb_model_flops(name.encode()))


def _torch():
    import torch
    return torch


class MpcbHandle:
    """One solver context: ``batch`` instances on the current CUDA device."""

    def __init__(self, library: MpcbLibrary, batch: int, opts_ss: Optional[Dict] = None,
                 opts_dyn: Optional[Dict] = None, device=None):
        torch = _torch()
        if not torch.cuda.is_available():
            raise RuntimeError("CUDA device required: the batched MPC solver has no CPU path")
        self.lib, self.L, self.batch = library, library.lib, int(batch)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        oss, ody = library.default_opts(), library.default_opts()
        for tgt, src in ((oss, opts_ss), (ody, opts_dyn)):
            for k, v in (src or {}).items():
                if not hasattr(tgt, k):
                    raise KeyError("unknown solver option %r" % k)
                setattr(tgt, k, v)
        self.opts_ss, self.opts_dyn = oss, ody
        self._h = ctypes.c_void_p()
        self.ocp_solves = 0             # OCP solves made through the handle (mpcb_ocp and the fused step): they reuse one workspace
        with torch.cuda.device(self.device):
            rc = self.L.mpcb_create(self.batch, ctypes.byref(oss), ctypes.byref(ody), ctypes.byref(self._h))
        self._check(rc)

    def _check(self, rc):
        if rc != 0:
            msg = self.L.mpcb_last_error(self._h)
            raise RuntimeError("mpcb error %d: %s" % (rc, msg.decode() if msg else "?"))

    def close(self):
        if self._h:
            self.L.mpcb_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- helpers ---------------------------------------------------------------
    def tensor(self, a, cols=None):
        """[B, cols] float64 tensor on the handle's device (broadcasts a single row over the batch)."""
        torch = _torch()
        t = a if isinstance(a, torch.Tensor) else torch.as_tensor(np.asarray(a, dtype=np.float64))
        t = t.to(device=self.device, dtype=torch.float64)
        if cols is not None:
            if t.ndim == 1:
                t = t.reshape(1, -1) if t.numel() == cols else t.reshape(-1, 1)
            if t.shape[0] == 1 and self.batch > 1:
                t = t.expand(self.batch, t.shape[1])
            if tuple(t.shape) != (self.batch, cols):
                raise ValueError("expected shape (%d, %d), got %s" % (self.batch, cols, tuple(t.shape)))
        return t.contiguous()

    def _stream(self):
        return ctypes.c_void_p(_torch().cuda.current_stream(self.device).cuda_stream)

    def empty(self, *shape, dtype=None):
        torch = _torch()
        return torch.empty(*shape, device=self.device, dtype=dtype or torch.float64)

    def set_const(self, name: str, values):
        v = np.ascontiguousarray(np.asarray(values, dtype=np.float64).reshape(-1))
        self._check(self.L.mpcb_set_const(self._h, name.encode(), v.ctypes.data, v.size))

    # -- entry points ------------------------------------------------------------
    def ocp(self, par, w):
        torch = _torch()
        d = self.lib.dims
        par = self.tensor(par, d.npar); w = self.tensor(w, d.nw).clone()
        f = self.empty(self.batch); st = self.empty(self.batch, dtype=torch.int32); it = self.empty(self.batch, dtype=torch.int32)
        self._check(self.L.mpcb_ocp(self._h, par.data_ptr(), w.data_ptr(), f.data_ptr(), st.data_ptr(), it.data_ptr(), self._stream()))
        self.ocp_solves += 1
        return w, f, st, it

    # -- sensitivities of the last OCP solve (include/mpcb.h, mpcb_ocp_sens_factor) -------------------------------
    @property
    def ntheta(self) -> int:
        d = self.lib.dims
        return 2 * (d.nx + d.nu)

    def ocp_sens_factor(self, par):
        """Capture of the sensitivities of the last `ocp` solve (``par`` must be that call's): ``(fac [B, size], status [B])``."""
        torch = _torch()
        par = self.tensor(par, self.lib.dims.npar)
        fac = self.empty(self.batch, int(self.L.mpcb_ocp_sens_size()))
        st = self.empty(self.batch, dtype=torch.int32)
        self._check(self.L.mpcb_ocp_sens_factor(self._h, par.data_ptr(), fac.data_ptr(), st.data_ptr(), self._stream()))
        return fac, st

    def ocp_jvp(self, fac, dtheta):
        """dw [B, ndir, nw] = J dtheta for dtheta [B, ndir, ntheta] (or [B, ntheta]: one direction)."""
        d = self.lib.dims
        dt = self.tensor(dtheta)
        if dt.ndim == 2:
            dt = dt.unsqueeze(1)
        if dt.ndim != 3 or dt.shape[0] != self.batch or dt.shape[2] != self.ntheta:
            raise ValueError("dtheta must be [B, ndir, %d], got %s" % (self.ntheta, tuple(dt.shape)))
        dt = dt.contiguous()
        dw = self.empty(self.batch, dt.shape[1], d.nw)
        self._check(self.L.mpcb_ocp_jvp(self._h, fac.data_ptr(), int(dt.shape[1]), dt.data_ptr(), dw.data_ptr(), self._stream()))
        return dw

    def ocp_vjp(self, fac, gw):
        """gtheta [B, ntheta] = J' gw for gw [B, nw]."""
        gw = self.tensor(gw, self.lib.dims.nw)
        g = self.empty(self.batch, self.ntheta)
        self._check(self.L.mpcb_ocp_vjp(self._h, fac.data_ptr(), gw.data_ptr(), g.data_ptr(), self._stream()))
        return g

    # -- sensitivities with respect to p = [d | px | py] (include/mpcb.h, mpcb_ocp_sens_factor_p) --------------------
    @property
    def np_params(self) -> int:
        d = self.lib.dims
        return d.nd + (d.npx + d.npy) * d.N

    def ocp_sens_factor_p(self, par):
        """As `ocp_sens_factor`, with the derivative blocks of p: ``(fac [B, size_p], status [B])``.  ``fac`` is one
        buffer of B * size_p doubles: the B theta captures (which the theta methods accept) followed by the p-blocks."""
        torch = _torch()
        par = self.tensor(par, self.lib.dims.npar)
        fac = self.empty(self.batch, int(self.L.mpcb_ocp_sens_size_p()))
        st = self.empty(self.batch, dtype=torch.int32)
        self._check(self.L.mpcb_ocp_sens_factor_p(self._h, par.data_ptr(), fac.data_ptr(), st.data_ptr(), self._stream()))
        return fac, st

    def _p_capture(self, fac):
        if fac.numel() != self.batch * int(self.L.mpcb_ocp_sens_size_p()):
            raise ValueError("the p sweeps need a capture of ocp_sens_factor_p")

    def ocp_jvp_p(self, fac, dp):
        """dw [B, ndir, nw] = J_p dp for dp [B, ndir, n_p] (or [B, n_p]: one direction)."""
        self._p_capture(fac)
        d = self.lib.dims
        dt = self.tensor(dp)
        if dt.ndim == 2:
            dt = dt.unsqueeze(1)
        if dt.ndim != 3 or dt.shape[0] != self.batch or dt.shape[2] != self.np_params:
            raise ValueError("dp must be [B, ndir, %d], got %s" % (self.np_params, tuple(dt.shape)))
        dt = dt.contiguous()
        dw = self.empty(self.batch, dt.shape[1], d.nw)
        self._check(self.L.mpcb_ocp_jvp_p(self._h, fac.data_ptr(), int(dt.shape[1]), dt.data_ptr(), dw.data_ptr(), self._stream()))
        return dw

    def ocp_vjp_p(self, fac, gw):
        """gp [B, n_p] = J_p' gw for gw [B, nw]."""
        self._p_capture(fac)
        gw = self.tensor(gw, self.lib.dims.nw)
        g = self.empty(self.batch, self.np_params)
        self._check(self.L.mpcb_ocp_vjp_p(self._h, fac.data_ptr(), gw.data_ptr(), g.data_ptr(), self._stream()))
        return g

    def target(self, par_ss, wss):
        torch = _torch()
        d = self.lib.dims
        par_ss = self.tensor(par_ss, d.nparss); wss = self.tensor(wss, d.nwss).clone()
        f = self.empty(self.batch); st = self.empty(self.batch, dtype=torch.int32); it = self.empty(self.batch, dtype=torch.int32)
        self._check(self.L.mpcb_target(self._h, par_ss.data_ptr(), wss.data_ptr(), f.data_ptr(), st.data_ptr(), it.data_ptr(), self._stream()))
        return wss, f, st, it

    # -- sensitivities of the target solution (include/mpcb.h, mpcb_target_sens_factor) ----------------------------
    @property
    def ntheta_ss(self) -> int:
        """Size of theta_ss = [usp | ysp | xsp | d | Us_prev | px | py]."""
        d = self.lib.dims
        return 2 * d.nu + d.ny + d.nx + d.nd + d.npx + d.npy

    def target_sens_factor(self, par_ss, wss0):
        """Capture of the sensitivities of the target solve from ``par_ss`` and the initial guess ``wss0`` (those of the
        `target` call; the problem is solved again): ``(fac [B, size], status [B])``."""
        torch = _torch()
        d = self.lib.dims
        par_ss = self.tensor(par_ss, d.nparss); wss0 = self.tensor(wss0, d.nwss)
        size = int(self.L.mpcb_target_sens_size())
        fac = self.empty(self.batch, max(size, 1))
        st = self.empty(self.batch, dtype=torch.int32)
        self._check(self.L.mpcb_target_sens_factor(self._h, par_ss.data_ptr(), wss0.data_ptr(), fac.data_ptr(), st.data_ptr(),
                                                   self._stream()))
        return fac, st

    def target_jvp(self, fac, dth):
        """dwss [B, ndir, nwss] = T dth for dth [B, ndir, ntheta_ss] (or [B, ntheta_ss]: one direction)."""
        d = self.lib.dims
        dt = self.tensor(dth)
        if dt.ndim == 2:
            dt = dt.unsqueeze(1)
        if dt.ndim != 3 or dt.shape[0] != self.batch or dt.shape[2] != self.ntheta_ss:
            raise ValueError("dth must be [B, ndir, %d], got %s" % (self.ntheta_ss, tuple(dt.shape)))
        dt = dt.contiguous()
        dw = self.empty(self.batch, dt.shape[1], d.nwss)
        self._check(self.L.mpcb_target_jvp(self._h, fac.data_ptr(), int(dt.shape[1]), dt.data_ptr(), dw.data_ptr(), self._stream()))
        return dw

    def target_vjp(self, fac, gw):
        """gth [B, ntheta_ss] = T' gw for gw [B, nwss]."""
        gw = self.tensor(gw, self.lib.dims.nwss)
        g = self.empty(self.batch, self.ntheta_ss)
        self._check(self.L.mpcb_target_vjp(self._h, fac.data_ptr(), gw.data_ptr(), g.data_ptr(), self._stream()))
        return g

    def estimate(self, est_type, y, u_prev, t, px, py, xi, P):
        d = self.lib.dims
        y = self.tensor(y, d.ny); u_prev = self.tensor(u_prev, d.nu); t = self.tensor(t, 1)
        px = self.tensor(px, d.npx); py = self.tensor(py, d.npy)
        xi = self.tensor(xi, d.nxi).clone(); P = self.tensor(P, d.nxi * d.nxi).clone()
        self._check(self.L.mpcb_estimate(self._h, int(est_type), y.data_ptr(), u_prev.data_ptr(), t.data_ptr(), px.data_ptr(),
                                         py.data_ptr(), xi.data_ptr(), P.data_ptr(), self._stream()))
        return xi, P

    def model_output(self, x, u, dd, t, py):
        d = self.lib.dims
        x = self.tensor(x, d.nx); u = self.tensor(u, d.nu); dd = self.tensor(dd, max(d.nd, 1)) if d.nd else self.empty(self.batch, 1)
        t = self.tensor(t, 1); py = self.tensor(py, d.npy)
        y = self.empty(self.batch, d.ny)
        self._check(self.L.mpcb_model_output(self._h, x.data_ptr(), u.data_ptr(), dd.data_ptr(), t.data_ptr(), py.data_ptr(), y.data_ptr(), self._stream()))
        return y

    def model_step(self, x, u, dd, t, px):
        d = self.lib.dims
        x = self.tensor(x, d.nx); u = self.tensor(u, d.nu); dd = self.tensor(dd, max(d.nd, 1)) if d.nd else self.empty(self.batch, 1)
        t = self.tensor(t, 1); px = self.tensor(px, d.npx)
        xn = self.empty(self.batch, d.nx)
        self._check(self.L.mpcb_model_step(self._h, x.data_ptr(), u.data_ptr(), dd.data_ptr(), t.data_ptr(), px.data_ptr(), xn.data_ptr(), self._stream()))
        return xn

    def plant_meas(self, x, u, t, pyp, pymp, noise=None):
        d = self.lib.dims
        x = self.tensor(x, d.nxp); u = self.tensor(u, d.nu); t = self.tensor(t, 1)
        pyp = self.tensor(pyp, d.npyp); pymp = self.tensor(pymp, d.npyp)
        nz = self.tensor(noise, d.ny) if noise is not None else None
        y = self.empty(self.batch, d.ny)
        self._check(self.L.mpcb_plant_meas(self._h, x.data_ptr(), u.data_ptr(), t.data_ptr(), pyp.data_ptr(), pymp.data_ptr(),
                                           nz.data_ptr() if nz is not None else None, y.data_ptr(), self._stream()))
        return y

    def plant_step(self, x, u, t, pxp, pxmp):
        d = self.lib.dims
        x = self.tensor(x, d.nxp).clone(); u = self.tensor(u, d.nu); t = self.tensor(t, 1)
        pxp = self.tensor(pxp, d.npxp); pxmp = self.tensor(pxmp, d.npxp)
        self._check(self.L.mpcb_plant_step(self._h, x.data_ptr(), u.data_ptr(), t.data_ptr(), pxp.data_ptr(), pxmp.data_ptr(), self._stream()))
        return x

    def stage_derivs(self, par, w, lam):
        d = self.lib.dims
        nz = d.nx + d.nu
        par = self.tensor(par, d.npar); w = self.tensor(w, d.nw); lam = self.tensor(lam, d.N * d.nx)
        A = self.empty(self.batch, d.N, d.nx * d.nx); Bm = self.empty(self.batch, d.N, d.nx * d.nu)
        c = self.empty(self.batch, d.N, d.nx); H = self.empty(self.batch, d.N, nz * (nz + 1) // 2)
        self._check(self.L.mpcb_stage_derivs(self._h, par.data_ptr(), w.data_ptr(), lam.data_ptr(), A.data_ptr(), Bm.data_ptr(),
                                             c.data_ptr(), H.data_ptr(), self._stream()))
        return A, Bm, c, H

    # -- fused closed-loop step ---------------------------------------------------
    def loop_reset(self, x0_m, u0, dhat0=None, P0=None):
        d = self.lib.dims
        x0_m = self.tensor(x0_m, d.nx); u0 = self.tensor(u0, d.nu)
        dh = self.tensor(dhat0, d.nd) if (dhat0 is not None and d.nd) else None
        P0 = self.tensor(P0, d.nxi * d.nxi) if P0 is not None else None
        _torch().cuda.current_stream(self.device).synchronize()
        self._check(self.L.mpcb_loop_reset(self._h, x0_m.data_ptr(), u0.data_ptr(), dh.data_ptr() if dh is not None else None,
                                           P0.data_ptr() if P0 is not None else None))
        torch = _torch()
        B = self.batch
        self._step_out = dict(u=self.empty(B, d.nu), xhat=self.empty(B, d.nx), dhat=self.empty(B, max(d.nd, 1)),
                              xs=self.empty(B, d.nx), us=self.empty(B, d.nu), f=self.empty(B),
                              status=self.empty(B, dtype=torch.int32), iters=self.empty(B, dtype=torch.int32),
                              status_ss=self.empty(B, dtype=torch.int32))

    def step(self, est_type, y_meas, t, sp, px=None, py=None):
        """One fused step; returns the dict of output tensors (reused between calls - clone to keep)."""
        d = self.lib.dims
        y = self.tensor(y_meas, d.ny); t = self.tensor(t, 1); sp = self.tensor(sp, d.nu + d.ny + d.nx)
        px = self.tensor(px, d.npx * d.N) if px is not None else None
        py = self.tensor(py, d.npy * d.N) if py is not None else None
        o = self._step_out
        self.ocp_solves += 1
        self._check(self.L.mpcb_step(self._h, int(est_type), y.data_ptr(), t.data_ptr(), sp.data_ptr(),
                                     px.data_ptr() if px is not None else None, py.data_ptr() if py is not None else None,
                                     o["u"].data_ptr(), o["xhat"].data_ptr(), o["dhat"].data_ptr(), o["xs"].data_ptr(),
                                     o["us"].data_ptr(), o["f"].data_ptr(), o["status"].data_ptr(), o["iters"].data_ptr(),
                                     o["status_ss"].data_ptr(), self._stream()))
        return o

    def set_groups(self, n: int):
        """Cut the batch of the fused step into ``n`` instance groups pipelined on separate streams (`mpcb_set_groups`)."""
        self._check(self.L.mpcb_set_groups(self._h, int(n)))

    def set_policy(self, hold_failed: bool):
        """Fused step: hold the previous input on every failed solve instead of applying its iterate (`mpcb_set_policy`)."""
        self._check(self.L.mpcb_set_policy(self._h, 1 if hold_failed else 0))

    def loop_state(self):
        """Copies of the device-resident loop state: xi = [x(k+1|k); d], P, u."""
        d = self.lib.dims
        xi, P, u = self.empty(self.batch, d.nxi), self.empty(self.batch, d.nxi * d.nxi), self.empty(self.batch, d.nu)
        self._check(self.L.mpcb_loop_get(self._h, xi.data_ptr(), P.data_ptr(), u.data_ptr(), self._stream()))
        return xi, P, u

    @property
    def last_ticks(self):
        """Solver ticks of the last OCP solve (waits for it: the count lives on the device)."""
        return self.L.mpcb_last_ticks(self._h)

    @property
    def launches(self):
        """Kernel launches made through this handle so far, the device-driven solver ticks included (synchronises)."""
        return int(self.L.mpcb_total_launches(self._h))

    KERNEL_CLASSES = ("ocp_init", "ocp_eval", "ocp_kkt", "ocp_trial", "ocp_accept", "target", "estimate", "other")

    def set_profiling(self, on: bool):
        self._check(self.L.mpcb_set_profiling(self._h, 1 if on else 0))

    def profile(self):
        """Accumulated CUDA-event time [ms] and launch count per kernel class since `set_profiling`."""
        ms = (ctypes.c_double * 8)(); ln = (ctypes.c_long * 8)(); cnt = (ctypes.c_ulonglong * 2)()
        self._check(self.L.mpcb_get_profile(self._h, ms, ln, cnt))
        return dict(ms=dict(zip(self.KERNEL_CLASSES, list(ms))), launches=dict(zip(self.KERNEL_CLASSES, list(ln))),
                    eval_instances=int(cnt[0]), trial_instances=int(cnt[1]))

    def dfma_peak_tflops(self, iters: int = 20000) -> float:
        out = ctypes.c_double(0.0)
        with _torch().cuda.device(self.device):
            rc = self.L.mpcb_dfma_peak(int(iters), ctypes.byref(out))
        if rc != 0:
            raise RuntimeError("mpcb_dfma_peak failed")
        return float(out.value)


class BatchedNlpSolver:
    """Stands in for the ``nlpsol`` object returned by the reference builders, for a batch of instances."""

    def __init__(self, kind: str, spec):
        if kind not in ("ocp", "target"):
            raise ValueError(kind)
        self.kind, self.spec = kind, spec
        self.handle: Optional[MpcbHandle] = None
        self._last = None
        self._last_ocp = None           # (par, handle solve count) of the last OCP call, for sensitivity()
        self._last_target = None        # copies of (p, x0) of the last target call, for sensitivity()
        self._bounds_key = None

    def attach(self, handle: MpcbHandle):
        self.handle = handle
        self._bounds_key = None
        return self

    def _require(self):
        if self.handle is None:
            raise RuntimeError("solver has no CUDA context: build one with mpc_code_b200.compile_problem(...) "
                               "(the solver runs only on the GPU; there is no CPU fallback)")

    def _push_bounds(self, lbx, ubx, lbg, ubg):
        s = self.spec
        lbx = s.w_lb if lbx is None else np.asarray(lbx, dtype=float)
        ubx = s.w_ub if ubx is None else np.asarray(ubx, dtype=float)
        lbg = s.g_lb if lbg is None else np.asarray(lbg, dtype=float)
        ubg = s.g_ub if ubg is None else np.asarray(ubg, dtype=float)
        if lbx.ndim == 2:   # per-instance rows: only the x0 block may differ, and that is taken from p
            lbx, ubx = lbx[0], ubx[0]
        lbx, ubx, lbg, ubg = [np.asarray(v, dtype=float).reshape(-1) for v in (lbx, ubx, lbg, ubg)]
        key = (lbx.tobytes(), ubx.tobytes(), lbg.tobytes(), ubg.tobytes())
        if key == self._bounds_key:
            return
        h = self.handle
        if self.kind == "ocp":
            n_dyn = s.n * (s.N + 1) + (s.n if s.term_eq is not None else 0)
            if np.any(lbg[:n_dyn] != 0.0) or np.any(ubg[:n_dyn] != 0.0):
                raise ValueError("the dynamics rows of g must stay equalities (lbg = ubg = 0)")
            h.set_const("ocp_lbx", lbx); h.set_const("ocp_ubx", ubx)
            # g = [dynamics | Y_k rows (all k) | DU_k rows (all k)]  (Control_Calc.py:200-204,254) -> stage-interleaved
            ny_rows = 0 if s.yFree else s.p * s.N
            ndu_rows = 0 if s.DuFree else s.m * s.N
            ngin_rows = s.n_gin * s.N
            def per_stage(v):
                blocks = []
                if ny_rows:
                    blocks.append(v[n_dyn:n_dyn + ny_rows].reshape(s.N, s.p))
                if ndu_rows:
                    blocks.append(v[n_dyn + ny_rows:n_dyn + ny_rows + ndu_rows].reshape(s.N, s.m))
                if ngin_rows:
                    o3 = n_dyn + ny_rows + ndu_rows
                    blocks.append(v[o3:o3 + ngin_rows].reshape(s.N, s.n_gin))
                return np.hstack(blocks).reshape(-1) if blocks else np.zeros(0)
            h.set_const("ocp_lbg", per_stage(lbg)); h.set_const("ocp_ubg", per_stage(ubg))
        else:
            if not (np.array_equal(lbg, s.g_lb) and np.array_equal(ubg, s.g_ub)):
                raise ValueError("the target problem's g bounds are fixed by its construction (Target_Calc.py:146-150): "
                                 "equalities, and -inf <= g_SS <= 0 for the user inequality rows")
            h.set_const("ss_lbx", lbx); h.set_const("ss_ubx", ubx)
        self._bounds_key = key

    def __call__(self, lbx=None, ubx=None, x0=None, p=None, lbg=None, ubg=None):
        self._require()
        self._push_bounds(lbx, ubx, lbg, ubg)
        if self.kind == "ocp":
            par = self.handle.tensor(p, self.handle.lib.dims.npar)
            x, f, st, it = self.handle.ocp(par, x0)
            self._last_ocp = (par, self.handle.ocp_solves)
        else:
            d = self.handle.lib.dims
            self._last_target = (self.handle.tensor(p, d.nparss).clone(), self.handle.tensor(x0, d.nwss).clone())
            x, f, st, it = self.handle.target(*self._last_target)
        self._last = (st, it)
        return {"x": x, "f": f}

    def sensitivity(self, params: bool = False):
        """Sensitivities of the last solve with respect to theta = [x_hat | x_s | u_s | u_{k-1}] (see
        `mpc_code_b200.sensitivity`): an `OcpSensitivity` that owns its capture and stays valid after later solves.
        ``params=True`` also captures the sensitivities with respect to p = [d | px | py] (`OcpSensitivity.jvp_p`).
        Must be called before the handle solves another OCP, with the solve's ``p`` not modified in place since.

        On the target solver: a `TargetSensitivity` of the last solve through this solver, with respect to theta_ss =
        [usp | ysp | xsp | d | Us_prev | px | py] (the problem is solved again from that call's ``p`` and ``x0``)."""
        if self.kind == "target":
            return self._target_sensitivity(params)
        self._require()
        if self._last_ocp is None:
            raise RuntimeError("sensitivity() before the first solve")
        par, solves = self._last_ocp
        if solves != self.handle.ocp_solves:
            raise RuntimeError("the handle has solved another OCP since this solver's last call: its workspace is gone")
        from .sensitivity import OcpSensitivity
        fac, st = (self.handle.ocp_sens_factor_p if params else self.handle.ocp_sens_factor)(par)
        return OcpSensitivity(self.handle, fac, st, uses_uprev=bool(self.spec.uses_uprev), params=params)

    def _target_sensitivity(self, params):
        if params:
            raise ValueError("params=True is for the OCP: theta_ss of the target problem already contains d, px and py")
        self._require()
        if self._last_target is None:
            raise NotImplementedError("sensitivity() of the target problem before a solve through this solver: the fused "
                                      "step (mpcb_step) keeps its target problem on the device and has no sensitivities")
        from .sensitivity import TargetSensitivity
        fac, st = self.handle.target_sens_factor(*self._last_target)
        return TargetSensitivity(self.handle, fac, st)

    def stats(self):
        if self._last is None:
            raise RuntimeError("stats() before the first solve")
        return _Stats(*self._last)


class _Stats(dict):
    """``solver.stats()``: ``status`` / ``iter_count`` are device tensors; ``return_status`` (IPOPT's strings, one per
    instance) and ``success`` need the codes on the host and are only fetched when asked for (a blocking copy)."""

    def __init__(self, status, iters):
        super().__init__(status=status, iter_count=iters)

    def __missing__(self, key):
        if key not in ("return_status", "success"):
            raise KeyError(key)
        codes = self["status"].cpu().numpy()
        self["return_status"] = [STATUS_NAMES.get(int(c), "Internal_Error") for c in codes]
        self["success"] = bool(np.all((codes == 0) | (codes == 1)))
        return dict.__getitem__(self, key)
