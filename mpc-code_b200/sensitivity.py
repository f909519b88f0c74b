"""Sensitivities of the batched OCP solution with respect to theta = [x_hat | x_s | u_s | u_{k-1}].

theta is the part of the OCP parameter vector that the closed loop feeds in from the estimator, the target problem and
the previous input: ``par[0 : 2nx+nu]`` and ``par[2nx+nu+nd : 2nx+2nu+nd]`` (``ntheta = 2 (nx + nu)``).  The
derivative is the implicit-function derivative of the barrier KKT system at the returned iterate (as sIPOPT computes
it, see ``include/mpcb.h``): strongly active bounds give derivatives of the order of the final barrier parameter.

The parameters that enter the dynamics, p = [d | px_0 .. px_{N-1} | py_0 .. py_{N-1}] = ``par[off_d : off_d+nd]`` ++
``par[off_px :]`` (``n_p = nd + (npx+npy) N``), have their own sensitivities (``sensitivity(params=True)``): the
disturbance estimate d_hat and the per-stage model offsets, whose derivatives are the controller's feed-forward gains.

* `OcpSensitivity` (from ``BatchedNlpSolver.sensitivity()``): JVP, VJP, the feedback gain dU_0/dx_hat and, with
  ``params=True``, the JVP / VJP in p and the disturbance gain dU_0/dd_hat.
* `OcpLayer`: the solve as a differentiable function of theta (and of p with ``params=True``) for ``torch.autograd``.

The steady-state target problem has sensitivities with respect to theta_ss = [usp | ysp | xsp | d | Us_prev | px | py],
the part of ``par_ss`` the loop feeds in (``par_ss`` without vec(lambda) and t; ``ntheta_ss = 2nu+ny+nx+nd+npx+npy``):

* `TargetSensitivity` (from ``solver_ss.sensitivity()``): JVP, VJP and the Jacobian dwss/dtheta_ss.
* `TargetLayer`: the target solve as a differentiable function of theta_ss.
* ``BatchedMpc.controller_gains()`` composes them with the OCP's into the controller's total gains.
"""
from __future__ import annotations


def _torch():
    import torch
    return torch


def theta_slices(nx: int, nu: int, nd: int):
    """The two slices of ``par`` that make up theta."""
    return slice(0, 2 * nx + nu), slice(2 * nx + nu + nd, 2 * nx + 2 * nu + nd)


def theta_of(par, nx: int, nu: int, nd: int):
    """theta [B, 2(nx+nu)] of OCP parameter vectors ``par`` [B, npar]."""
    a, b = theta_slices(nx, nu, nd)
    return _torch().cat([par[:, a], par[:, b]], dim=1)


def with_theta(par, theta, nx: int, nu: int, nd: int):
    """``par`` with its theta part replaced by ``theta`` (differentiable in both)."""
    a, b = theta_slices(nx, nu, nd)
    return _torch().cat([theta[:, :a.stop], par[:, a.stop:b.start], theta[:, a.stop:], par[:, b.stop:]], dim=1)


def param_slices(nx: int, nu: int, nd: int, ny: int):
    """The two slices of ``par`` that make up p = [d | px | py]: d, and everything from the offsets of px on."""
    off_d = 2 * nx + nu
    return slice(off_d, off_d + nd), slice(2 * nx + 2 * nu + nd + 1 + ny * nu, None)


def params_of(par, nx: int, nu: int, nd: int, ny: int):
    """p [B, n_p] of OCP parameter vectors ``par`` [B, npar]."""
    a, b = param_slices(nx, nu, nd, ny)
    return _torch().cat([par[:, a], par[:, b]], dim=1)


def with_params(par, p, nx: int, nu: int, nd: int, ny: int):
    """``par`` with its p part replaced by ``p`` (differentiable in both)."""
    a, b = param_slices(nx, nu, nd, ny)
    return _torch().cat([par[:, :a.start], p[:, :nd], par[:, a.stop:b.start], p[:, nd:]], dim=1)


class OcpSensitivity:
    """Captured sensitivities of one batched OCP solve.  ``status`` [B] (int32, device): 0 computed, 1 the solve ended
    with a status other than 0 / 1, 2 wrong inertia of the KKT matrix; every output of an instance with status != 0 is
    NaN.  The capture ``fac`` belongs to this object, so results do not change when the handle solves again."""

    def __init__(self, handle, fac, status, uses_uprev: bool, params: bool = False):
        self.handle, self.fac, self.status, self.uses_uprev, self.params = handle, fac, status, uses_uprev, params
        d = handle.lib.dims
        self.nx, self.nu, self.nd, self.ntheta = d.nx, d.nu, d.nd, handle.ntheta

    def jvp(self, dtheta):
        """dw [B, ndir, nw] for dtheta [B, ndir, ntheta]; a [B, ntheta] input gives [B, nw]."""
        dw = self.handle.ocp_jvp(self.fac, dtheta)
        return dw[:, 0] if getattr(dtheta, "ndim", 3) == 2 else dw

    def vjp(self, gw):
        """gtheta [B, ntheta] = (dw/dtheta)' gw for gw [B, nw]."""
        return self.handle.ocp_vjp(self.fac, gw)

    def feedback_gain(self):
        """dU_0/dx_hat [B, nu, nx], the local feedback law of the controller; with Delta-u terms (u_{k-1} carried as
        state) also dU_0/du_{k-1} [B, nu, nu], returned as a second tensor."""
        torch = _torch()
        nx, nu, B = self.nx, self.nu, self.handle.batch
        cols = list(range(nx)) + (list(range(2 * nx + nu, 2 * nx + 2 * nu)) if self.uses_uprev else [])
        E = torch.zeros(len(cols), self.ntheta, dtype=torch.float64, device=self.handle.device)
        E[torch.arange(len(cols)), torch.tensor(cols)] = 1.0
        dw = self.handle.ocp_jvp(self.fac, E.expand(B, -1, -1))
        du0 = dw[:, :, nx:nx + nu].transpose(1, 2).contiguous()          # [B, nu, ndir]
        return (du0[:, :, :nx].contiguous(), du0[:, :, nx:].contiguous()) if self.uses_uprev else du0

    def _require_params(self):
        if not self.params:
            raise RuntimeError("captured without the p-blocks: use solver.sensitivity(params=True)")

    def jvp_p(self, dp):
        """dw [B, ndir, nw] for dp [B, ndir, n_p], p = [d | px | py]; a [B, n_p] input gives [B, nw]."""
        self._require_params()
        dw = self.handle.ocp_jvp_p(self.fac, dp)
        return dw[:, 0] if getattr(dp, "ndim", 3) == 2 else dw

    def vjp_p(self, gw):
        """gp [B, n_p] = (dw/dp)' gw for gw [B, nw]."""
        self._require_params()
        return self.handle.ocp_vjp_p(self.fac, gw)

    def disturbance_gain(self):
        """dU_0/dd_hat [B, nu, nd] with the targets x_s, u_s held fixed: the OCP's response to the disturbance estimate.
        In the closed loop d_hat also moves x_s and u_s through the target problem; that part is not included here.
        ``BatchedMpc.controller_gains()["d_hat"]`` is the total derivative through the target problem."""
        self._require_params()
        torch = _torch()
        nx, nu, nd, B = self.nx, self.nu, self.nd, self.handle.batch
        E = torch.zeros(nd, self.handle.np_params, dtype=torch.float64, device=self.handle.device)
        E[torch.arange(nd), torch.arange(nd)] = 1.0
        dw = self.handle.ocp_jvp_p(self.fac, E.expand(B, -1, -1))
        return dw[:, :, nx:nx + nu].transpose(1, 2).contiguous()


def theta_ss_slices(nx: int, nu: int, ny: int, nd: int):
    """The two slices of ``par_ss`` that make up theta_ss: [usp | ysp | xsp | d | Us_prev], and [px | py]."""
    off_lam = 2 * nu + ny + nx + nd
    return slice(0, off_lam), slice(off_lam + ny * nu + 1, None)


def theta_ss_of(par_ss, nx: int, nu: int, ny: int, nd: int):
    """theta_ss [B, ntheta_ss] of target parameter vectors ``par_ss`` [B, nparss]."""
    a, b = theta_ss_slices(nx, nu, ny, nd)
    return _torch().cat([par_ss[:, a], par_ss[:, b]], dim=1)


def with_theta_ss(par_ss, theta_ss, nx: int, nu: int, ny: int, nd: int):
    """``par_ss`` with its theta_ss part replaced by ``theta_ss`` (differentiable in both)."""
    a, b = theta_ss_slices(nx, nu, ny, nd)
    return _torch().cat([theta_ss[:, :a.stop], par_ss[:, a.stop:b.start], theta_ss[:, a.stop:]], dim=1)


class TargetSensitivity:
    """Captured sensitivities of one batched target solve with respect to theta_ss.  ``status`` [B] (int32, device): 0
    computed, 1 the solve ended with a status other than 0 / 1, 2 wrong inertia of the KKT matrix; every output of an
    instance with status != 0 is NaN.  The capture ``fac`` belongs to this object."""

    def __init__(self, handle, fac, status):
        self.handle, self.fac, self.status = handle, fac, status
        self.ntheta_ss = handle.ntheta_ss

    @property
    def wss(self):
        """[B, nwss] the solution the capture was taken at (bit for bit the output of the target solve it repeats)."""
        return self.fac[:, 2:2 + self.handle.lib.dims.nwss]

    def jvp(self, dth):
        """dwss [B, ndir, nwss] for dth [B, ndir, ntheta_ss]; a [B, ntheta_ss] input gives [B, nwss]."""
        dw = self.handle.target_jvp(self.fac, dth)
        return dw[:, 0] if getattr(dth, "ndim", 3) == 2 else dw

    def vjp(self, gw):
        """gth [B, ntheta_ss] = (dwss/dtheta_ss)' gw for gw [B, nwss]."""
        return self.handle.target_vjp(self.fac, gw)

    def jacobian(self):
        """dwss/dtheta_ss [B, nwss, ntheta_ss]."""
        torch = _torch()
        E = torch.eye(self.ntheta_ss, dtype=torch.float64, device=self.handle.device)
        return self.handle.target_jvp(self.fac, E.expand(self.handle.batch, -1, -1)).transpose(1, 2).contiguous()


class TargetLayer:
    """``wss = TargetLayer(solver_ss)(theta_ss, par_ss, wss0)``: the batched target solve as a function of theta_ss,
    differentiable through ``torch.autograd`` (backward = one VJP on the captured factorisation).  ``par_ss`` supplies
    vec(lambda) and t (its theta_ss part is replaced) and ``wss0`` is the initial guess; neither may require grad.
    Once differentiable."""

    def __init__(self, solver_ss, lbx=None, ubx=None):
        if solver_ss.kind != "target":
            raise NotImplementedError("TargetLayer wraps the target solver")
        self.solver, self.bounds = solver_ss, dict(lbx=lbx, ubx=ubx)
        self.last = None                # TargetSensitivity of the last forward pass

    def __call__(self, theta_ss, par_ss, wss0):
        for name, t in (("par_ss", par_ss), ("wss0", wss0)):
            if getattr(t, "requires_grad", False):
                raise ValueError("TargetLayer differentiates with respect to theta_ss only: %s must not require grad "
                                 "(sensitivities with respect to t and lambda are not available)" % name)
        return _target_function().apply(theta_ss, par_ss, wss0, self)


class OcpLayer:
    """``w = OcpLayer(solver)(theta, par, w0)``: the batched OCP solve as a function of theta, differentiable through
    ``torch.autograd`` (backward = one VJP sweep on the captured factorisation).  theta is the only differentiable
    input: ``par`` supplies the other parameters (its theta part is replaced) and ``w0`` is the initial guess; neither
    may require grad.  Once differentiable (the backward pass is not itself differentiable).

    ``OcpLayer(solver, params=True)(theta, par, w0, p)``: p = [d | px | py] [B, n_p] is a second differentiable input
    (it replaces the p part of ``par``); the backward pass is still one sweep per input."""

    def __init__(self, solver, lbx=None, ubx=None, lbg=None, ubg=None, params: bool = False):
        if solver.kind != "ocp":
            raise NotImplementedError("OcpLayer wraps the dynamic OCP solver")
        self.solver, self.bounds, self.params = solver, dict(lbx=lbx, ubx=ubx, lbg=lbg, ubg=ubg), params
        self.last = None                # OcpSensitivity of the last forward pass

    def __call__(self, theta, par, w0, p=None):
        for name, t in (("par", par), ("w0", w0)):
            if getattr(t, "requires_grad", False):
                raise ValueError("OcpLayer differentiates with respect to theta%s only: %s must not require grad "
                                 "(sensitivities with respect to t and lambda are not available)"
                                 % (" and p" if self.params else " (and p with params=True)", name))
        if p is not None and not self.params:
            raise ValueError("p is a differentiable input only with OcpLayer(..., params=True)")
        if self.params and p is None:
            raise ValueError("OcpLayer(..., params=True) takes p [B, n_p] as its fourth input")
        if not self.params:
            return _ocp_function().apply(theta, par, w0, self)
        return _ocp_function_p().apply(theta, p, par, w0, self)


def _make_function():
    torch = _torch()
    from torch.autograd.function import once_differentiable

    class OcpFunction(torch.autograd.Function):
        @staticmethod
        def forward(ctx, theta, par, w0, layer):
            h = layer.solver.handle
            d = h.lib.dims
            p = with_theta(h.tensor(par, d.npar), theta.detach().to(h.device, torch.float64), d.nx, d.nu, d.nd)
            sol = layer.solver(x0=w0, p=p, **layer.bounds)
            sens = layer.solver.sensitivity()
            layer.last = sens
            ctx.sens = sens
            ctx.dtype, ctx.device = theta.dtype, theta.device
            return sol["x"]

        @staticmethod
        @once_differentiable
        def backward(ctx, gw):
            g = ctx.sens.vjp(gw.contiguous())
            return g.to(device=ctx.device, dtype=ctx.dtype), None, None, None

    return OcpFunction


def _make_function_p():
    torch = _torch()
    from torch.autograd.function import once_differentiable

    class OcpFunctionP(torch.autograd.Function):
        @staticmethod
        def forward(ctx, theta, p, par, w0, layer):
            h = layer.solver.handle
            d = h.lib.dims
            pt = with_theta(h.tensor(par, d.npar), theta.detach().to(h.device, torch.float64), d.nx, d.nu, d.nd)
            pt = with_params(pt, p.detach().to(h.device, torch.float64), d.nx, d.nu, d.nd, d.ny)
            sol = layer.solver(x0=w0, p=pt, **layer.bounds)
            sens = layer.solver.sensitivity(params=True)
            layer.last = sens
            ctx.sens = sens
            ctx.meta = (theta.dtype, theta.device, p.dtype, p.device)
            return sol["x"]

        @staticmethod
        @once_differentiable
        def backward(ctx, gw):
            gw = gw.contiguous()
            tdt, tdev, pdt, pdev = ctx.meta
            gth = ctx.sens.vjp(gw).to(device=tdev, dtype=tdt) if ctx.needs_input_grad[0] else None
            gp = ctx.sens.vjp_p(gw).to(device=pdev, dtype=pdt) if ctx.needs_input_grad[1] else None
            return gth, gp, None, None, None

    return OcpFunctionP


def _make_target_function():
    torch = _torch()
    from torch.autograd.function import once_differentiable

    class TargetFunction(torch.autograd.Function):
        @staticmethod
        def forward(ctx, theta_ss, par_ss, wss0, layer):
            h = layer.solver.handle
            d = h.lib.dims
            p = with_theta_ss(h.tensor(par_ss, d.nparss), theta_ss.detach().to(h.device, torch.float64), d.nx, d.nu, d.ny, d.nd)
            sol = layer.solver(x0=wss0, p=p, **layer.bounds)
            sens = layer.solver.sensitivity()
            layer.last = sens
            ctx.sens = sens
            ctx.dtype, ctx.device = theta_ss.dtype, theta_ss.device
            return sol["x"]

        @staticmethod
        @once_differentiable
        def backward(ctx, gw):
            g = ctx.sens.vjp(gw.contiguous())
            return g.to(device=ctx.device, dtype=ctx.dtype), None, None, None

    return TargetFunction


_FUNCTION = None
_FUNCTION_P = None
_FUNCTION_TGT = None


def _target_function():
    global _FUNCTION_TGT
    if _FUNCTION_TGT is None:
        _FUNCTION_TGT = _make_target_function()
    return _FUNCTION_TGT


def _ocp_function():
    """The autograd Function, defined on first use (the package imports torch lazily)."""
    global _FUNCTION
    if _FUNCTION is None:
        _FUNCTION = _make_function()
    return _FUNCTION


def _ocp_function_p():
    global _FUNCTION_P
    if _FUNCTION_P is None:
        _FUNCTION_P = _make_function_p()
    return _FUNCTION_P
