"""Batched closed loop: the body of the reference driver's ``for ksim`` loop, for B instances at once.

Statement by statement this is ``MPC_code.py:485-875`` (estimator dispatch ``:546-668``, target
``:690-731``, OCP warm start / solve / extraction ``:734-810``, plant step ``:813-827``) with every
per-instance quantity turned into a ``[B, n]`` CUDA tensor and the CasADi calls replaced by the
batched solver objects.  Results keep the reference's names (``Xp, Yp, U, XS, US, YS, X_HAT,
Y_HAT, D_HAT, TIME_SS, TIME_DYN``).  Measurement noise is an explicit ``[Nsim, B, ny]`` input
(the reference draws it from an unseeded global RNG, ``:538-541``).
"""
from __future__ import annotations

import os
import time
from typing import Dict, Optional

import numpy as np

from .build import build_library
from .control_calc import opt_dyn  # noqa: F401  (re-exported: reference-compatible builder names)
from .loader import load_example
from .problem import MpcProblem, build_problem, make_specs
from .solvers import BatchedNlpSolver, MpcbHandle, MpcbLibrary
from .target_calc import opt_ss  # noqa: F401

INFEASIBLE = 2


class CompiledProblem:
    """A problem whose CUDA library is built and loaded; factory for per-batch controllers."""

    def __init__(self, prob: MpcProblem, name: str = "problem", verbose: bool = False):
        self.prob, self.name = prob, name
        self.ss_spec, self.ocp_spec = make_specs(prob)
        self.build = build_library(name, prob, self.ss_spec, self.ocp_spec, verbose=verbose)
        self.library = MpcbLibrary(self.build["so"])
        self.flops = self.build["gen"]["flops"]

    def controller(self, batch: int, opts_ss: Optional[Dict] = None, opts_dyn: Optional[Dict] = None, device=None,
                   hold_on_failure: bool = False):
        return BatchedMpc(self, batch, opts_ss, opts_dyn, device, hold_on_failure)


def compile_problem(example, name: Optional[str] = None, overrides: Optional[Dict] = None, verbose=False) -> CompiledProblem:
    """``example``: path of an ``Ex_*.py``-style file, a loaded namespace, or an `MpcProblem`."""
    if isinstance(example, MpcProblem):
        prob = example
    else:
        ns = load_example(example, overrides) if isinstance(example, (str, os.PathLike)) else example
        prob = build_problem(ns)
        if name is None and isinstance(example, (str, os.PathLike)):
            name = os.path.splitext(os.path.basename(str(example)))[0]
    return CompiledProblem(prob, (name or "problem").lower(), verbose=verbose)


def torch_where_failed(t, st, hold):
    """Status as the warm-start gate sees it: with the hold policy a failed solve counts as infeasible."""
    return t.where((st < 0) & (st != -13), t.full_like(st, INFEASIBLE), st) if hold else st


class BatchedMpc:
    """Loop state of B instances plus the solver objects; ``step()`` is one pass of the hot path."""

    def __init__(self, cp: CompiledProblem, batch: int, opts_ss=None, opts_dyn=None, device=None, hold_on_failure: bool = False):
        """``hold_on_failure``: treat every FAILED OCP solve (iteration limit, restoration failed, ...) like an infeasible
        one - previous input kept, estimate propagated by the model.  Default False = the reference, which only rejects
        'Infeasible_Problem_Detected' (``MPC_code.py:786``)."""
        import torch
        self.torch = torch
        self.cp, self.prob, self.B = cp, cp.prob, int(batch)
        p = self.prob
        itmax = p.sol_optss["ipopt.max_iter"]
        oss = dict(max_iter=itmax); oss.update(opts_ss or {})
        ody = dict(max_iter=p.sol_optdyn["ipopt.max_iter"]); ody.update(opts_dyn or {})
        self.h = MpcbHandle(cp.library, self.B, oss, ody, device)
        self.hold_on_failure = bool(hold_on_failure)
        self.h.set_policy(self.hold_on_failure)
        self.solver_ss = BatchedNlpSolver("target", cp.ss_spec).attach(self.h)
        self.solver = BatchedNlpSolver("ocp", cp.ocp_spec).attach(self.h)
        est = p.estimator
        self.est_type = 0 if est["type"] == "kalss" else 1
        if self.est_type == 0:
            self.h.set_const("K_est", est["K"])
        else:
            self.h.set_const("Q_kf", est["Q"]); self.h.set_const("R_kf", est["R"])
        if (est["dmin"] is not None or est["dmax"] is not None) and p.nd:      # one-sided bounds: the other side is open
            self.h.set_const("dmin", est["dmin"] if est["dmin"] is not None else np.full(p.nd, -np.inf))
            self.h.set_const("dmax", est["dmax"] if est["dmax"] is not None else np.full(p.nd, np.inf))
        self.reset()

    # -- state -----------------------------------------------------------------
    def _rows(self, v, n):
        return self.h.tensor(np.asarray(v, dtype=float).reshape(1, n) if np.ndim(v) < 2 else v, n).clone()

    def reset(self, x0_p=None, x0_m=None, u0=None, dhat0=None):
        """Initial loop state (``MPC_code.py:442-463``); each may be one row or ``[B, n]``."""
        p, t = self.prob, self.torch
        self.x_k = self._rows(p.x0_p if x0_p is None else x0_p, p.nxp)
        self.x0_m = self._rows(p.x0_m if x0_m is None else x0_m, p.nx)
        self.u0 = self._rows(p.u0 if u0 is None else u0, p.nu)
        self.u_k = self.u0.clone()
        self.xhat_k = self.x0_m.clone()
        self.dhat_k = self._rows(p.dhat0 if dhat0 is None else dhat0, max(p.nd, 1)) if p.nd else self.h.empty(self.B, 0)
        self.P_k = self._rows(p.estimator["P0"].reshape(1, -1), p.nxi * p.nxi)
        self.lam = t.zeros(self.B, p.ny * p.nu, device=self.h.device, dtype=t.float64)
        self.us_k = self.u_k.clone(); self.xs_k = self.x0_m.clone()
        self.w_opt = None; self.w_guess = None
        self.dyn_status = t.zeros(self.B, dtype=t.int32, device=self.h.device)
        self.dead = t.zeros(self.B, dtype=t.bool, device=self.h.device)
        self._fused = False
        self.x_k0, self.dhat0, self.P0 = self.x_k.clone(), self.dhat_k.clone(), self.P_k.clone()
        self.ksim = 0

    def _bury(self, bad):
        """The reference exits the process when a state turns NaN (``MPC_code.py:671-673,819-821``).  In a batch
        one diverged instance must not stop the others: it is flagged in ``dead`` and re-seeded with the nominal
        initial state so that the kernels keep receiving finite numbers; its outputs are meaningless from then on."""
        if not bool(bad.any()):
            return
        t = self.torch
        self.dead |= bad
        m = bad.unsqueeze(1)
        self.x_k = t.where(m, self.x_k0, self.x_k)
        self.xhat_k = t.where(m, self.x0_m, self.xhat_k)
        self.u_k = t.where(m, self.u0, self.u_k)
        if self.prob.nd:
            self.dhat_k = t.where(m, self.dhat0, self.dhat_k)
        self.P_k = t.where(m, self.P0, self.P_k)

    def _row(self, v, slot=None):
        """``[B, n]`` device tensor holding the host vector ``v`` in every row.  With ``slot`` the tensor is cached by value:
        the host-side parameter vectors are constant in most problems, and an upload from pageable host memory synchronises
        the stream, which would stop the host from enqueueing the next step ahead of the GPU."""
        t = self.torch
        a = np.ascontiguousarray(np.asarray(v, dtype=float).reshape(1, -1))
        if slot is None:
            return t.as_tensor(a, device=self.h.device).expand(self.B, -1).contiguous()
        cache = self.__dict__.setdefault("_row_cache", {})
        key = a.tobytes()
        hit = cache.get(slot)
        if hit is None or hit[0] != key:
            hit = (key, t.as_tensor(a, device=self.h.device).expand(self.B, -1).contiguous())
            cache[slot] = hit
        return hit[1]

    def _params(self, t_k):
        """Time-varying parameters along the horizon (``MPC_code.py:492-515``)."""
        p, ns = self.prob, self.prob.ns
        p_xk = np.zeros((p.npx, p.N)); p_yk = np.zeros((p.npy, p.N))
        if "def_px" in ns:
            for i in range(p.N):
                p_xk[:, i] = np.asarray(ns["def_px"](t_k + i)[0], dtype=float).ravel()
        if "def_py" in ns:
            for i in range(p.N):
                p_yk[:, i] = np.asarray(ns["def_py"](t_k + i)[0], dtype=float).ravel()
        p_xmp = np.zeros(p.npxp); p_ymp = np.zeros(p.npyp)
        if "def_px" in ns:
            p_xmp = np.asarray(ns["def_pxmp"](t_k)[0], dtype=float).ravel() if "def_pxmp" in ns else p_xk[:, 0].copy()
        if "def_py" in ns:
            p_ymp = np.asarray(ns["def_pymp"](t_k)[0], dtype=float).ravel() if "def_pymp" in ns else p_yk[:, 0].copy()
        p_xp = np.asarray(ns["def_pxp"](t_k)[0], dtype=float).ravel() if "def_pxp" in ns else np.zeros(p.npxp)
        p_yp = np.asarray(ns["def_pyp"](t_k)[0], dtype=float).ravel() if "def_pyp" in ns else np.zeros(p.npyp)
        return p_xk, p_yk, p_xmp, p_ymp, p_xp, p_yp

    # -- one closed-loop step -----------------------------------------------------
    def step(self, noise=None, state_noise=None, time_phases: bool = False, y_meas=None) -> Dict[str, object]:
        """One closed-loop step.  With ``y_meas`` (``[B, ny]``) the measurement comes from the caller (a real
        plant) and the built-in plant simulation (``MPC_code.py:531-541,813-827``) is skipped."""
        p, t, h = self.prob, self.torch, self.h
        nx, nu, ny, nd, N, B = p.nx, p.nu, p.ny, p.nd, p.N, self.B
        nxu = nx + nu
        dev, f64 = h.device, t.float64
        t_k = self.ksim * p.h
        tt = t.full((B, 1), t_k, device=dev, dtype=f64)
        p_xk, p_yk, p_xmp, p_ymp, p_xp, p_yp = self._params(t_k)
        row = self._row
        p_x_k, p_y_k = row(p_xk[:, 0]), row(p_yk[:, 0])
        out: Dict[str, object] = dict(Xp=self.x_k.clone(), X_HAT=self.xhat_k.clone())
        nominal = p.flags["Fp_nominal"] is True
        offree = p.flags["offree"]
        # model and plant outputs (:524-541)
        yhat_k = h.model_output(self.xhat_k, self.u_k, self.dhat_k, tt, p_y_k)
        if y_meas is not None:
            y_k = h.tensor(y_meas, ny)
        elif nominal:
            y_k = h.model_output(self.x_k, self.u_k, self.dhat_k, tt, p_y_k)
            if noise is not None:
                y_k = y_k + h.tensor(noise, ny)
        else:
            y_k = h.plant_meas(self.x_k, self.u_k, tt, row(p_yp), row(p_ymp), noise)
        out["Yp"], out["Y_HAT"] = y_k, yhat_k
        # estimator (:546-668)
        xi = t.cat([self.xhat_k, self.dhat_k], dim=1) if offree != "no" else self.xhat_k
        xi, self.P_k = h.estimate(self.est_type, y_k, self.u_k, tt, p_x_k, p_y_k, xi, self.P_k)
        if offree != "no":
            self.xhat_k, self.dhat_k = xi[:, :nx].contiguous(), xi[:, nx:].contiguous()
        else:
            self.xhat_k = xi
        out["D_HAT"] = self.dhat_k.clone()
        self._bury(t.isnan(self.xhat_k).any(dim=1) | (t.isnan(self.dhat_k).any(dim=1) if nd else False))   # :671-673
        if p.flags["estimating"] is False:
            if p.defSP is not None:
                ysp_k, usp_k, xsp_k = [row(v) for v in p.defSP(t_k)]
            else:
                ysp_k, usp_k, xsp_k = [t.zeros(B, n_, device=dev, dtype=f64) for n_ in (ny, nu, nx)]
            us_prev, xs_prev = self.us_k.clone(), self.xs_k.clone()
            par_ss = t.cat([usp_k, ysp_k, xsp_k, self.dhat_k, us_prev, self.lam, tt, p_x_k, p_y_k], dim=1)   # :693
            y0 = h.model_output(self.x0_m, self.u0, self.dhat_k, tt, p_y_k)
            wss_guess = t.cat([self.x0_m, self.u0, y0], dim=1)                                               # :696-700
            if time_phases:
                t.cuda.synchronize(dev); t0 = time.time()
            sol_ss = self.solver_ss(lbx=None, ubx=None, x0=wss_guess, p=par_ss, lbg=None, ubg=None)          # :704-709
            if time_phases:
                t.cuda.synchronize(dev); out["TIME_SS"] = time.time() - t0
            st_ss = self.solver_ss.stats()["status"]
            ok = (st_ss != INFEASIBLE).unsqueeze(1)                                                         # :714-718
            wss = sol_ss["x"]
            self.xs_k = t.where(ok, wss[:, :nx], self.xs_k)
            self.us_k = t.where(ok, wss[:, nx:nxu], self.us_k)
            out["XS"], out["US"] = self.xs_k.clone(), self.us_k.clone()
            out["YS"] = h.model_output(self.xs_k, self.us_k, self.dhat_k, tt, p_y_k)                        # :730
            out["STATUS_SS"], out["ITER_SS"], out["F_SS"] = st_ss, self.solver_ss.stats()["iter_count"], sol_ss["f"]
            # warm start (:740-764)
            if self.ksim == 0:
                stage = t.cat([self.x0_m, self.u0], dim=1)
                self.w_guess = t.cat([stage.repeat(1, N), self.x0_m], dim=1)
            else:
                shifted = t.cat([self.w_opt[:, nxu:], us_prev, xs_prev], dim=1)
                keep = (self.dyn_status == INFEASIBLE).unsqueeze(1)
                self.w_guess = t.where(keep, self.w_guess, shifted)
            par = t.cat([self.xhat_k, self.xs_k, self.us_k, self.dhat_k, self.u_k, tt, self.lam,
                         row(p_xk.reshape(-1, order="F")), row(p_yk.reshape(-1, order="F"))], dim=1)         # :769-772
            if time_phases:
                t.cuda.synchronize(dev); t0 = time.time()
            sol = self.solver(lbx=None, ubx=None, x0=self.w_guess, p=par, lbg=None, ubg=None)                # :776-781
            if time_phases:
                t.cuda.synchronize(dev); out["TIME_DYN"] = time.time() - t0
            st = self.solver.stats()["status"]
            self.dyn_status = torch_where_failed(t, st, self.hold_on_failure)
            okd = (st != INFEASIBLE) & (st != -13)                           # :786-805; a NaN iterate (-13) is never adopted
            if self.hold_on_failure:
                okd = okd & (st >= 0)
            okd = okd.unsqueeze(1)
            w_new = sol["x"]
            self.w_opt = w_new if self.w_opt is None else t.where(okd, w_new, self.w_opt)
            x_pred = h.model_step(self.xhat_k, self.u_k, self.dhat_k, tt, p_x_k)
            self.xhat_k = t.where(okd, w_new[:, nxu:nxu + nx], x_pred)
            self.u_k = t.where(okd, w_new[:, nx:nxu], self.u_k)
            out["U"] = self.u_k.clone()
            out["STATUS_DYN"], out["ITER_DYN"], out["F_DYN"] = st, self.solver.stats()["iter_count"], sol["f"]
        # plant step (:813-827)
        if y_meas is not None:
            self.ksim += 1
            return out
        if nominal:
            self.x_k = h.model_step(self.x_k, self.u_k, self.dhat_k, tt, row(p_xmp))
        else:
            self.x_k = h.plant_step(self.x_k, self.u_k, tt, row(p_xp, "pxp"), row(p_xmp, "pxmp"))
        if state_noise is not None:
            self.x_k = self.x_k + h.tensor(state_noise, p.nxp)
        self._bury(t.isnan(self.x_k).any(dim=1))                                                           # :819-821
        out["DEAD"] = self.dead.clone()
        self.ksim += 1
        return out

    def feedback_gain(self):
        """Local feedback law of the controller at the last `step()`: dU_0/dx_hat [B, nu, nx] of that step's OCP solve
        (with Delta-u terms also dU_0/du_{k-1}, see `OcpSensitivity.feedback_gain`).  Not available after
        `step_fused`, whose OCP parameters stay on the device."""
        if self._fused:
            raise RuntimeError("feedback_gain() after step_fused(): the fused step keeps its OCP parameters on the device; "
                               "use step()")
        return self.solver.sensitivity().feedback_gain()

    def controller_gains(self):
        """The controller's linearisation at the last `step()`, through the target problem and the OCP: a dict of
        [B, nu, n] tensors

        * ``x_hat``: dU_0/dx_hat (the target does not read x_hat: `feedback_gain`);
        * ``u_prev``: dU_0/du_{k-1} with Delta-u terms, else None;
        * ``usp``, ``ysp``, ``xsp``: the set-point gains J_theta[:, x_s|u_s] T[(x_s,u_s), .] with T = dwss/dtheta_ss;
        * ``d_hat``: the total dU_0/dd_hat = J_p[:, d] + J_theta[:, x_s|u_s] T[(x_s,u_s), d]; None when nd = 0 or when the
          OCP has no sensitivities with respect to p (decided at code generation).

        An instance whose target solve was rejected as infeasible keeps its previous targets, so its T-terms are zero;
        an instance whose OCP or target capture failed gives NaN.  Not available after `step_fused`."""
        if self._fused:
            raise RuntimeError("controller_gains() after step_fused(): the fused step keeps its target and OCP problems on "
                               "the device; use step()")
        t, p = self.torch, self.prob
        nx, nu, ny, nd = p.nx, p.nu, p.ny, p.nd
        with_p = bool(nd) and bool(self.cp.build["gen"]["defines"].get("MPCB_SENS_P"))
        ocp = self.solver.sensitivity(params=with_p)
        K = ocp.feedback_gain()
        out = dict(x_hat=K[0], u_prev=K[1]) if self.cp.ocp_spec.uses_uprev else dict(x_hat=K, u_prev=None)
        # dU_0/d[x_s; u_s]: theta columns nx .. 2nx+nu
        E = t.zeros(nx + nu, self.h.ntheta, dtype=t.float64, device=self.h.device)
        E[t.arange(nx + nu), t.arange(nx, 2 * nx + nu)] = 1.0
        G = ocp.jvp(E.expand(self.B, -1, -1))[:, :, nx:nx + nu].transpose(1, 2)              # [B, nu, nx+nu]
        T = self.solver_ss.sensitivity().jacobian()[:, :nx + nu]                               # [B, nx+nu, ntheta_ss]
        T = T.masked_fill((self.solver_ss.stats()["status"] == INFEASIBLE).view(-1, 1, 1), 0.0)
        GT = t.bmm(G, T)                                                                      # [B, nu, ntheta_ss]
        for name, a, n in (("usp", 0, nu), ("ysp", nu, ny), ("xsp", nu + ny, nx)):
            out[name] = GT[:, :, a:a + n].contiguous()
        o_d = nu + ny + nx
        out["d_hat"] = ocp.disturbance_gain() + GT[:, :, o_d:o_d + nd] if with_p else None
        return out

    # -- the same step through the fused C entry point (mpcb_step): no host glue between the solves ----------
    def fused_reset(self):
        """Hand the current loop state to the device-resident loop of `mpcb_step`.  Only at the start of a run: the
        device loop keeps more state than is handed over here (previous targets, warm start, the first-step flag)."""
        if self.ksim > 0:
            raise RuntimeError("fused_reset after %d step() calls: switch between step() and step_fused() only after reset()" % self.ksim)
        self.solver_ss._push_bounds(None, None, None, None)      # w_lb/w_ub/g_lb/g_ub of the builders -> device constants
        self.solver._push_bounds(None, None, None, None)
        self.h.loop_reset(self.xhat_k, self.u_k, self.dhat_k if self.prob.nd else None, self.P_k)
        self._fused = True

    def step_fused(self, noise=None, y_meas=None, record_prediction: bool = False) -> Dict[str, object]:
        """One closed-loop step with estimator, target, OCP and extraction done by `mpcb_step`.  Same semantics and
        results as `step` (tests compare them); only the plant simulation and the set-point lookup stay on the host."""
        if not getattr(self, "_fused", False):
            self.fused_reset()
        p, t, h = self.prob, self.torch, self.h
        B, dev, f64 = self.B, h.device, t.float64
        t_k = self.ksim * p.h
        if getattr(self, "_tt", None) is None:
            self._tt = t.empty(B, 1, device=dev, dtype=f64)
        self._tt.fill_(t_k)
        tt = self._tt
        p_xk, p_yk, p_xmp, p_ymp, p_xp, p_yp = self._params(t_k)
        row = self._row
        varying = any(k in p.ns for k in ("def_px", "def_py"))
        px = row(p_xk.reshape(-1, order="F"), "px") if varying else None
        py = row(p_yk.reshape(-1, order="F"), "py") if varying else None
        out: Dict[str, object] = {}
        if record_prediction:                               # x(k|k-1) as the reference logs it (MPC_code.py:520)
            out["X_HAT"] = h.loop_state()[0][:, :p.nx].contiguous()
        if y_meas is None:
            out["Xp"] = self.x_k.clone()
            if p.flags["Fp_nominal"] is True:
                raise NotImplementedError("fused step with a nominal plant: pass y_meas")
            y_meas = h.plant_meas(self.x_k, self.u_k, tt, row(p_yp, "pyp"), row(p_ymp, "pymp"), noise)
            simulate = True
        else:
            simulate = False
        out["Yp"] = y_meas
        sp_key = t_k if p.defSP is not None else None
        if getattr(self, "_sp_key", object()) != sp_key or getattr(self, "_sp", None) is None:
            vals = p.defSP(t_k) if p.defSP is not None else (np.zeros(p.ny), np.zeros(p.nu), np.zeros(p.nx))
            ysp, usp, xsp = [np.asarray(v, dtype=float).ravel() for v in vals]
            self._sp = row(np.concatenate([usp, ysp, xsp]), "sp"); self._sp_key = sp_key     # uploaded only when the values change
        o = h.step(self.est_type, y_meas, tt, self._sp, px, py)
        self.u_k = o["u"]
        self.dead |= o["status"] == -13          # Invalid_Number_Detected: diverged instance, frozen (MPC_code.py:671-673 exits)
        out.update(U=o["u"], X_CORR=o["xhat"], D_HAT=o["dhat"], XS=o["xs"], US=o["us"], F_DYN=o["f"],
                   STATUS_DYN=o["status"], ITER_DYN=o["iters"], STATUS_SS=o["status_ss"])
        if simulate:
            self.x_k = h.plant_step(self.x_k, self.u_k, tt, row(p_xp, "pxp"), row(p_xmp, "pxmp"))
        self.ksim += 1
        return out

    def run(self, Nsim: Optional[int] = None, noise=None, state_noise=None, fused: bool = False) -> Dict[str, object]:
        """Run ``Nsim`` steps and stack the per-step records into ``[Nsim, B, n]`` tensors (``MPC_code.py:877-895``)."""
        t = self.torch
        Nsim = self.prob.Nsim if Nsim is None else Nsim
        if fused and state_noise is not None:
            raise NotImplementedError("state noise is not applied by the fused step: use fused=False")
        rec: Dict[str, list] = {}
        for k in range(Nsim):
            if fused:
                o = {key: (val.clone() if isinstance(val, t.Tensor) else val)
                     for key, val in self.step_fused(None if noise is None else noise[k], record_prediction=True).items()}
            else:
                o = self.step(None if noise is None else noise[k], None if state_noise is None else state_noise[k])
            for key, val in o.items():
                rec.setdefault(key, []).append(val)
        return {k: t.stack([t.as_tensor(x) for x in v]) for k, v in rec.items()}
