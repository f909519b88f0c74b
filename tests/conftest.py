import ctypes
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import mpc_code_b200  # noqa: E402,F401
import __graft_entry__ as entry  # noqa: E402

REFERENCE = os.environ.get("MPC_CODE_REFERENCE", "")     # an unmodified CPCLAB-UNIPI/MPC-code checkout, if any
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        have_gpu = torch.cuda.is_available()
    except Exception:
        have_gpu = False
    if have_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


class Bundle:
    """Problem + specs + oracle model + (lazily) the CPU harness / CUDA library of one example."""

    def __init__(self, name):
        from mpc_code_b200.build import build_library
        self.name = name
        self.prob, self.ss, self.ocp = entry._problem(name)
        self._oracle = self._harness = self._lib = None
        self._build_library = build_library

    @property
    def oracle(self):
        if self._oracle is None:
            from oracle import cmodel
            self._oracle = cmodel.build(self.name, self.prob, self.ocp, self.ss)
        return self._oracle

    @property
    def lib(self):
        if self._lib is None:
            self._lib = self._build_library(self.name, self.prob, self.ss, self.ocp)
        return self._lib

    @property
    def harness(self):
        if self._harness is None:
            res = self.lib
            path = entry.harness_path(res, self.name)
            if not os.path.exists(path):
                entry.build_harness(os.path.dirname(res["header"]), path)
            self._harness = ctypes.CDLL(path)
        return self._harness

    # ---- conveniences for the CSTR-style tests ---------------------------------
    def ocp_par(self, xhat, xs, us, d, um1=None, t=0.0):
        p = self.prob
        um1 = p.u0 if um1 is None else um1
        return np.concatenate([xhat, xs, us, d, um1, [t], np.zeros(p.ny * p.nu),
                               np.zeros(p.npx * p.N), np.zeros(p.npy * p.N)])

    def cold_guess(self):
        p = self.prob
        nxu = p.nx + p.nu
        w = np.zeros(p.nw)
        for k in range(p.N + 1):
            w[nxu * k:nxu * k + p.nx] = p.x0_m
        for k in range(p.N):
            w[nxu * k + p.nx:nxu * (k + 1)] = p.u0
        return w

    def ocp_range_bounds(self):
        """Range rows of g_lb/g_ub stage by stage: [Y_k bounds, DU_k bounds] for k = 0..N-1 (see include/mpcb.h)."""
        o = self.ocp
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

    def harness_ocp(self, par, w0, max_iter=100, tol=1e-8, mu_init=0.1, relax=1e-8, honor=0):
        H = self.harness
        par = np.ascontiguousarray(np.atleast_2d(par), dtype=float); w = np.ascontiguousarray(np.atleast_2d(w0), dtype=float).copy()
        B = par.shape[0]
        f = np.zeros(B); st = np.zeros(B, dtype=np.int32); it = np.zeros(B, dtype=np.int32); ticks = ctypes.c_int(0)
        lbg, ubg = self.ocp_range_bounds()
        if lbg.size == 0:
            lbg = ubg = np.zeros(1)
        lbx, ubx = np.ascontiguousarray(self.ocp.w_lb), np.ascontiguousarray(self.ocp.w_ub)
        H.h_ocp.argtypes = [ctypes.c_int] + [ctypes.c_void_p] * 9 + [ctypes.c_int, ctypes.c_double, ctypes.c_double,
                                                                     ctypes.c_double, ctypes.c_int, ctypes.c_void_p]
        H.h_ocp(B, par.ctypes.data, w.ctypes.data, f.ctypes.data, st.ctypes.data, it.ctypes.data, lbx.ctypes.data,
                ubx.ctypes.data, lbg.ctypes.data, ubg.ctypes.data, max_iter, tol, mu_init, relax, honor, ctypes.addressof(ticks))
        return w, f, st, it, ticks.value

    def harness_target(self, par, w0, max_iter=100):
        H = self.harness
        par = np.ascontiguousarray(np.atleast_2d(par), dtype=float); w = np.ascontiguousarray(np.atleast_2d(w0), dtype=float).copy()
        B = par.shape[0]
        f = np.zeros(B); st = np.zeros(B, dtype=np.int32); it = np.zeros(B, dtype=np.int32)
        lbx, ubx = np.ascontiguousarray(self.ss.w_lb), np.ascontiguousarray(self.ss.w_ub)
        H.h_target.argtypes = [ctypes.c_int] + [ctypes.c_void_p] * 7 + [ctypes.c_int, ctypes.c_double, ctypes.c_double,
                                                                        ctypes.c_double, ctypes.c_int]
        H.h_target(B, par.ctypes.data, w.ctypes.data, f.ctypes.data, st.ctypes.data, it.ctypes.data, lbx.ctypes.data,
                   ubx.ctypes.data, max_iter, 1e-8, 0.1, 1e-8, 0)
        return w, f, st, it


_BUNDLES = {}


def _bundle(name):
    if name not in _BUNDLES:
        _BUNDLES[name] = Bundle(name)
    return _BUNDLES[name]


@pytest.fixture(scope="session")
def nmpc():
    return _bundle("nmpc_cstr")


@pytest.fixture(scope="session")
def lmpc_cstr():
    return _bundle("lmpc_cstr")


@pytest.fixture(scope="session")
def lmpc_wb():
    return _bundle("lmpc_wb")


@pytest.fixture(scope="session")
def enmpc():
    return _bundle("enmpc_reactor")


@pytest.fixture(scope="session")
def lmpc_nlplant():
    return _bundle("lmpc_nlplant")


@pytest.fixture(scope="session")
def nmpc_dis():
    return _bundle("nmpc_dis")


@pytest.fixture(scope="session")
def lmpcxp_nlplant():
    return _bundle("lmpcxp_nlplant")
