"""The OCP solve under every build-time kernel mapping the sources keep, and the mappings they refuse.

The KKT kernel (and the sensitivity factor, which shares its mapping) runs on MPCB_KKT_LANES = 32 lanes per instance by
default; -DMPCB_KKT_LANES=1/16/8/4 are one thread per instance and lane groups.  The evaluation kernel has its own
switches (MPCB_EVAL_FIRST, MPCB_STAGE_CACHE, MPCB_EVAL_SMEM, MPCB_VEC_REC).  Each of these is a different device code
path; the `-m gpu` tests below build every one listed in PLAN and compare it with the default build of the same problem
on the same inputs.  Without a GPU: the refusals, and the CPU harness without the stage cache.
"""
import ctypes
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import __graft_entry__ as entry
from conftest import GOLDEN, ROOT, Bundle, _bundle

G = np.load(os.path.join(GOLDEN, "nmpc_oracle.npz"))


def _build(name, flags):
    from mpc_code_b200.build import build_library
    prob, ss, ocp = entry._problem(name)
    return build_library(name, prob, ss, ocp, extra_flags=flags)


# ==== refusals: stop in the compiler's front end, with a message that names the switch ================================
LANES_MSG = "MPCB_KKT_LANES must be one of 1, 2, 4, 8, 16, 32"
SMEM_MSG = "exceeds the 48 kB of static shared memory"


@pytest.mark.parametrize("name, flags, message", [
    ("nmpc_cstr", ("-DMPCB_KKT_LANES=12",), LANES_MSG),
    ("nmpc_cstr", ("-DMPCB_KKT_LANES=64",), LANES_MSG),
    ("syn_12_4_20", ("-DMPCB_KKT_LANES=4",), SMEM_MSG),                     # 8 scratches of 2 510 doubles per warp
    ("syn_20_6_20", ("-DMPCB_KKT_LANES=16",), SMEM_MSG),
], ids=["lanes12", "lanes64", "syn_12_4_20-lanes4", "syn_20_6_20-lanes16"])
def test_unsupported_mapping_is_refused_at_compile_time(name, flags, message):
    with pytest.raises(RuntimeError, match="nvcc failed") as err:
        _build(name, flags)
    assert message in str(err.value)


# ==== the CPU harness without the stage cache: the generator's uncached functions (Sys::f, not f_rc) ==================
STAGE_CACHE0 = ("-DMPCB_STAGE_CACHE=0",)


class _UncachedBundle(Bundle):
    """A bundle whose CPU harness is compiled with -DMPCB_STAGE_CACHE=0."""

    @property
    def harness(self):
        if self._harness is None:
            from mpc_code_b200.build import build_dir_for
            res = self.lib
            path = entry.harness_path(res, self.name + "_stage_cache0")
            path = os.path.join(build_dir_for(os.path.dirname(path), os.path.basename(path)), os.path.basename(path))
            if not os.path.exists(path):
                os.makedirs(os.path.dirname(path), exist_ok=True)
                entry.build_harness(os.path.dirname(res["header"]), path, flags=STAGE_CACHE0)
            self._harness = ctypes.CDLL(path)
        return self._harness


def test_harness_without_stage_cache_matches_oracle_fixtures():
    """Ex_NMPC (one cached transcendental, two reciprocals per stage point): the golden OCP batch, the infeasible start
    and the closed loop of tests/test_device_cpu.py, with the same bounds."""
    from harness_loop import HarnessLoop
    nmpc = _UncachedBundle("nmpc_cstr")
    assert nmpc.lib["gen"]["defines"]["MPCB_MDL_NC"] > 0      # otherwise the switch changes nothing
    par, w0 = G["ocp_par"], np.tile(G["ocp_w0"], (G["ocp_par"].shape[0], 1))
    w, f, st, it, _ = nmpc.harness_ocp(par, w0)
    assert np.array_equal(st, G["ocp_status"]) and np.array_equal(it, G["ocp_iters"])
    assert np.abs(w - G["ocp_w"]).max() < 1e-9
    assert np.all(np.abs(f - G["ocp_f"]) <= 1e-10 * np.maximum(1.0, np.abs(G["ocp_f"])))
    p = nmpc.prob
    xhat = p.x0_m.copy(); xhat[2] = 0.4995
    _, _, st, it, _ = nmpc.harness_ocp(nmpc.ocp_par(xhat, p.x0_m, p.u0, p.dhat0), nmpc.cold_guess())
    assert st[0] == 2 and it[0] == 0
    rec = HarnessLoop(nmpc, G["cl_x0"].shape[0]).run(G["cl_noise"].shape[0], G["cl_x0"], G["cl_noise"])
    assert np.array_equal(rec["STATUS_DYN"], G["cl_STATUS_DYN"]) and np.array_equal(rec["ITER_DYN"], G["cl_ITER_DYN"])
    for key in ("U", "X_HAT", "D_HAT", "XS", "US", "Xp", "Yp"):
        assert np.abs(rec[key] - G["cl_" + key]).max() < 1e-6, key
    assert np.all(np.abs(rec["F_DYN"] - G["cl_F_DYN"]) <= 1e-8 * np.maximum(1.0, np.abs(G["cl_F_DYN"])))


def test_harness_without_stage_cache_matches_the_cached_one():
    """The four-state synthetic plant (four cached tanh per stage point, N = 70): same statuses and iterations, w to
    rounding.  (enmpc_reactor has no stage cache, so the switch does not change its code.)"""
    from test_synthetic import _cases
    b, bu = _bundle("syn_4_2_70"), _UncachedBundle("syn_4_2_70")
    assert b.lib["gen"]["defines"]["MPCB_MDL_NC"] > 0
    par, w0 = _cases(b, 5)
    w, f, st, it, _ = b.harness_ocp(par, w0)
    wu, fu, stu, itu, _ = bu.harness_ocp(par, w0)
    assert np.all(st == 0) and np.array_equal(st, stu) and np.array_equal(it, itu)
    assert np.all(np.abs(wu - w) <= 1e-9 * np.maximum(1.0, np.abs(w)))
    assert np.all(np.abs(fu - f) <= 1e-10 * np.maximum(1.0, np.abs(f)))


# ==== on the device: every mapping against the default build ==========================================================
BITWISE, TOLERANCE = "bitwise", "tolerance"
# The first-tick kernel adds the multiplier terms as exact zeros, but it takes x+, A and B from dyn_sens, a separately
# compiled forward sweep whose FMA contraction differs from dyn_full's: equal to rounding, not bit for bit (a host build
# with -ffp-contract=fast differs by one ulp at a third of the stage points; without contraction they are identical).
# Without the stage cache the right-hand side is other generated expressions, again contracted differently on the
# device.  One Ex_NMPC instance of the batch has an ill-conditioned capture (its barrier derivative is 1e-3 away from
# the active-set one), which turns those roundings into 2e-8 of its columns: hence 1e-7 for that mapping's capture.
MAPPINGS = {   # label: (nvcc flags, comparison class with the default build, rtol of the captured columns)
    "lanes1": (("-DMPCB_KKT_LANES=1",), TOLERANCE, 1e-9),    # reductions in another order
    "lanes16": (("-DMPCB_KKT_LANES=16",), TOLERANCE, 1e-9),
    "lanes8": (("-DMPCB_KKT_LANES=8",), TOLERANCE, 1e-9),
    "lanes4": (("-DMPCB_KKT_LANES=4",), TOLERANCE, 1e-9),
    "evalfirst0": (("-DMPCB_EVAL_FIRST=0",), TOLERANCE, 1e-9),
    "stagecache0": (("-DMPCB_STAGE_CACHE=0",), TOLERANCE, 1e-7),
    "evalsmem0": (("-DMPCB_EVAL_SMEM=0",), BITWISE, 0.0),    # sub-step records in local memory
    "vecrec0": (("-DMPCB_VEC_REC=0",), BITWISE, 0.0),        # scalar record stores
}
KKT = ("lanes1", "lanes16", "lanes8", "lanes4")
PLAN = {   # problem: the mappings it is checked under (those that change its code and build)
    "nmpc_cstr": KKT + ("evalfirst0", "stagecache0", "evalsmem0", "vecrec0"),   # RK4, output rows, first-tick kernel
    "nmpc_cstr_termcons": KKT,                   # terminal equality: Pi / Gramian scratch, FREC_GA terms
    "lmpc_wb": KKT,                              # Delta-u form: NXA > NX
    "enmpc_reactor": KKT + ("evalsmem0", "vecrec0"),   # ContForm, indefinite Hessian: early sweep exit, restoration
    "syn_4_2_70": KKT,                           # N = 70: several rounds of every stage loop at every lane count
    "syn_20_6_20": ("lanes1",),                  # KKT_NBUF = 2, dense derivative path; lane groups do not fit
}
ROWS = [(name, label) for name, labels in PLAN.items() for label in labels]
ROW_IDS = ["%s-%s" % row for row in ROWS]
B = 37                                           # ragged for every lane-group size


_BUILD_ONE = ("import sys, __graft_entry__ as e\n"
              "from mpc_code_b200.build import build_library\n"
              "name, flags = sys.argv[1], tuple(sys.argv[2:])\n"
              "build_library(name, *e._problem(name), extra_flags=flags)\n")


@pytest.fixture(scope="module")
def libraries():
    """Build the default and every listed mapping of each problem once, in parallel nvcc processes (the code generator
    keeps module state, so each build runs in its own interpreter).  A failed build fails its rows, not the module."""
    env = dict(os.environ)
    env.pop("MPCB_EXTRA_FLAGS", None)
    jobs = [(name, ()) for name in PLAN] + [(name, MAPPINGS[label][0]) for name, label in ROWS]
    jobs.sort(key=lambda j: not j[0].startswith("syn_20"))          # the longest builds first
    python = [sys.executable] + (["-s"] if sys.flags.no_user_site else [])

    def run(job):
        subprocess.run(python + ["-c", _BUILD_ONE, job[0], *job[1]], cwd=ROOT, env=env, capture_output=True)
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as pool:
        list(pool.map(run, jobs))


_COMPILED = {}


def _compiled(name, flags):
    from mpc_code_b200.mpc_loop import CompiledProblem
    if (name, flags) not in _COMPILED:
        with pytest.MonkeyPatch.context() as mp:
            mp.setenv("MPCB_EXTRA_FLAGS", " ".join(flags))
            _COMPILED[(name, flags)] = CompiledProblem(_bundle(name).prob, name)
    return _COMPILED[(name, flags)]


def _batch(name):
    """B parameter vectors and the initial guess: seeded perturbations as in tests/test_ocp_sensitivity.py."""
    from test_ocp_sensitivity import sample_pars
    b = _bundle(name)
    p = b.prob
    rng = np.random.default_rng(37)
    if name == "nmpc_cstr":       # the golden instances, perturbed; an infeasible start (status 2 at iteration 0) in the middle
        par = G["ocp_par"][np.arange(B) % G["ocp_par"].shape[0]].copy()
        par[:, :2 * p.nx] *= 1 + 0.002 * rng.uniform(-1, 1, (B, 2 * p.nx))
        xhat = p.x0_m.copy(); xhat[2] = 0.4995
        par[B // 2] = b.ocp_par(xhat, p.x0_m, p.u0, p.dhat0)
        return par, G["ocp_w0"]
    if name.startswith("syn_"):
        return np.stack([b.ocp_par(rng.uniform(-1, 1, p.nx), np.zeros(p.nx), np.zeros(p.nu), np.zeros(0))
                         for _ in range(B)]), np.zeros(p.nw)
    return sample_pars(b, B, seed=37), b.cold_guess()


def _solve_and_capture(cp, par, w0):
    """One batched solve, then the theta capture: status, jvp(eye) and vjp(gw)."""
    import torch
    from mpc_code_b200.solvers import BatchedNlpSolver, MpcbHandle
    n, nw = par.shape[0], cp.prob.nw
    h = MpcbHandle(cp.library, n, dict(max_iter=100), dict(max_iter=100))
    solver = BatchedNlpSolver("ocp", cp.ocp_spec).attach(h)
    sol = solver(x0=np.ascontiguousarray(np.broadcast_to(w0, (n, nw))), p=par)
    stats = solver.stats()
    sens = solver.sensitivity()
    nth = h.ntheta
    dw = sens.jvp(torch.eye(nth, dtype=torch.float64, device=h.device).expand(n, -1, -1))
    gw = np.random.default_rng(2).standard_normal((n, nw))
    gth = sens.vjp(gw)
    out = dict(w=sol["x"], f=sol["f"], status=stats["status"], iters=stats["iter_count"], sstatus=sens.status, dw=dw, gth=gth)
    return {k: v.cpu().numpy() for k, v in out.items()}


def _closed_loop(cp, name):
    """Six steps of the fused step from seeded plant states (Ex_ENMPC: its restoration start on every other instance)."""
    p = cp.prob
    rng = np.random.default_rng(6)
    if name == "enmpc_reactor":
        from test_edge_cases import _enmpc_hard_start
        x0 = np.clip(np.array([0.9, 0.1]) + 0.05 * rng.uniform(-1, 1, (B, p.nxp)), 0.0, 1.0)
        x0[::2] = _enmpc_hard_start(_bundle(name))
        x0_m = np.tile(p.x0_m, (B, 1))
    elif name.startswith("syn_"):
        x0 = x0_m = rng.uniform(-1, 1, (B, p.nx))
    else:
        x0 = x0_m = p.x0_p * (1 + 0.02 * rng.uniform(-1, 1, (B, p.nxp)))
    ctl = cp.controller(B)
    ctl.reset(x0_p=x0, x0_m=x0_m)
    return {k: v.cpu().numpy() for k, v in ctl.run(6, fused=True).items()}


_DEFAULT = {}


def _default(kind, name):
    if (kind, name) not in _DEFAULT:
        cp = _compiled(name, ())
        _DEFAULT[(kind, name)] = _solve_and_capture(cp, *_batch(name)) if kind == "solve" else _closed_loop(cp, name)
    return _DEFAULT[(kind, name)]


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.int64) if a.dtype == np.float64 else a


def _rel_dev(a, r):
    """max |a - r| / max(1, |r|) over the finite entries (NaN patterns are compared separately)."""
    ok = np.isfinite(r)
    return float((np.abs(a[ok] - r[ok]) / np.maximum(1.0, np.abs(r[ok]))).max(initial=0.0))


def _assert_bitwise(got, ref):
    for key in ref:
        assert got[key].shape == ref[key].shape and np.array_equal(_bits(got[key]), _bits(ref[key])), \
            "%s differs: max |d| = %.3e" % (key, np.nanmax(np.abs(got[key].astype(float) - ref[key].astype(float))))


@pytest.mark.gpu
@pytest.mark.parametrize("name, label", ROWS, ids=ROW_IDS)
def test_batch_solve_and_theta_capture_match_the_default_build(libraries, name, label, record_property):
    flags, cls, rtol = MAPPINGS[label]
    par, w0 = _batch(name)
    ref = _default("solve", name)
    assert (ref["sstatus"] == 0).sum() >= B // 2                   # the capture comparison is not vacuous
    if name == "nmpc_cstr":
        assert ref["status"][B // 2] == 2 and ref["iters"][B // 2] == 0 and ref["sstatus"][B // 2] == 1
    got = _solve_and_capture(_compiled(name, flags), par, w0)
    if cls == BITWISE:
        _assert_bitwise(got, ref)
        record_property("max_dev", "bitwise")
        return
    for key in ("status", "iters", "sstatus"):
        assert np.array_equal(got[key], ref[key]), key
    dev_w, dev_f = _rel_dev(got["w"], ref["w"]), _rel_dev(got["f"], ref["f"])
    assert dev_w <= 1e-9 and dev_f <= 1e-10, (dev_w, dev_f)
    ok = ref["sstatus"] == 0
    assert np.all(np.isnan(got["dw"][~ok])) and np.all(np.isnan(got["gth"][~ok]))
    from test_ocp_sensitivity import _col_close
    dev_s = 0.0
    for i in np.where(ok)[0]:
        R, A = ref["dw"][i].T, got["dw"][i].T                      # [nw, ntheta]
        assert np.all(_col_close(A, R, rtol)), (i, np.abs(A - R).max(axis=0))
        scale = np.maximum(np.abs(R).max(axis=0), 1e-3 * max(np.abs(R).max(), 1e-300))
        dev_s = max(dev_s, float((np.abs(A - R).max(axis=0) / scale).max()))
        g, gr = got["gth"][i], ref["gth"][i]
        assert np.allclose(g, gr, rtol=rtol, atol=rtol * np.abs(gr).max()), (i, np.abs(g - gr).max())
    record_property("max_dev", "w %.1e f %.1e sens %.1e" % (dev_w, dev_f, dev_s))


@pytest.mark.gpu
@pytest.mark.parametrize("name, label", ROWS, ids=ROW_IDS)
def test_fused_closed_loop_matches_the_default_build(libraries, name, label, record_property):
    flags, cls, _ = MAPPINGS[label]
    ref = _default("loop", name)
    got = _closed_loop(_compiled(name, flags), name)
    assert set(got) == set(ref)
    if cls == BITWISE:
        _assert_bitwise(got, ref)
        record_property("max_dev", "bitwise")
        return
    dev = 0.0
    for key in ref:
        if ref[key].dtype.kind in "iub":
            assert np.array_equal(got[key], ref[key]), key
            continue
        assert np.array_equal(np.isnan(got[key]), np.isnan(ref[key])), key
        d = _rel_dev(got[key], ref[key])
        assert d <= (1e-10 if key == "F_DYN" else 1e-9), (key, d)
        dev = max(dev, d)
    record_property("max_dev", "%.1e" % dev)


@pytest.mark.gpu
@pytest.mark.parametrize("label", PLAN["nmpc_cstr"])
def test_golden_batch_matches_oracle_fixtures(libraries, nmpc, label):
    """The absolute anchor of every Ex_NMPC mapping: the tolerances of tests/test_gpu_parity.py."""
    from mpc_code_b200.solvers import BatchedNlpSolver, MpcbHandle
    cp = _compiled("nmpc_cstr", MAPPINGS[label][0])
    n = G["ocp_par"].shape[0]
    h = MpcbHandle(cp.library, n, dict(max_iter=100), dict(max_iter=100))
    solver = BatchedNlpSolver("ocp", cp.ocp_spec).attach(h)
    sol = solver(lbx=nmpc.ocp.w_lb, ubx=nmpc.ocp.w_ub, x0=np.tile(G["ocp_w0"], (n, 1)), p=G["ocp_par"],
                 lbg=nmpc.ocp.g_lb, ubg=nmpc.ocp.g_ub)
    w, f = sol["x"].cpu().numpy(), sol["f"].cpu().numpy()
    stats = solver.stats()
    assert np.array_equal(stats["status"].cpu().numpy(), G["ocp_status"])
    assert np.array_equal(stats["iter_count"].cpu().numpy(), G["ocp_iters"])
    assert np.abs(w - G["ocp_w"]).max() < 1e-8
    assert np.all(np.abs(f - G["ocp_f"]) <= 1e-8 * np.maximum(1.0, np.abs(G["ocp_f"])))
