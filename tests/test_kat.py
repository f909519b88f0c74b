"""Known-answer facts derivable from the reference's own example constants (SURVEY.md section 4)."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, REFERENCE
from mpc_code_b200.loader import load_example
from mpc_code_b200.problem import build_problem, make_specs
from mpc_code_b200.sx import Function, jacobian

KAT = json.load(open(os.path.join(GOLDEN, "kat.json")))


def test_kat1_example_initial_point_is_a_steady_state(nmpc):
    p = nmpc.prob
    k1 = KAT["KAT1"]
    assert np.allclose(p.x0_m, k1["x0_m"]) and np.allclose(p.u0, k1["u0"]) and np.allclose(p.dhat0, k1["dhat0"])
    f = np.asarray(p.Fx_model.meta["rhs"](p.x0_m, p.u0, p.dhat0, 0.0, np.zeros(3))).ravel()
    assert np.allclose(f, k1["f_expected"], atol=3e-5, rtol=0.05)
    res = np.asarray(p.Fx_model(p.x0_m, p.u0, p.h, p.dhat0, 0.0, np.zeros(3))).ravel() - p.x0_m
    assert np.allclose(res, k1["rk4_residual_expected"], atol=1e-5, rtol=0.05)


def test_kat2_rk4_jacobians_match_the_linearisation_printed_in_the_reference(nmpc):
    """Ex_LMPC_nlplant.py:85-91 prints A, B of the RK4 (10 sub-steps, h=0.2) CSTR map at (xlin, ulin), F0 = 0.1."""
    p, k2 = nmpc.prob, KAT["KAT2"]
    s = p.sym
    assert p.h == k2["h"] and p.Fx_p.meta["substeps"] == k2["Mx"]
    Fp = p.Fx_p(s["xp"], s["u"], s["pxp"], s["t"], s["k"], s["pxmp"])
    JA = Function("JA", [s["xp"], s["u"], s["pxp"], s["t"], s["k"], s["pxmp"]], [jacobian(Fp, s["xp"]), jacobian(Fp, s["u"])])
    A, B = JA(np.array(k2["xlin"]), np.array(k2["ulin"]), np.zeros(3), 0.0, k2["h"], np.zeros(3))   # t=0 -> F0 = 0.1
    assert np.abs(np.asarray(A) - np.array(k2["A"])).max() < 6e-5      # six printed digits of 53.6817
    assert np.abs(np.asarray(B) - np.array(k2["B"])).max() < 6e-6


def test_kat3_target_solutions_of_the_oracle(nmpc):
    from oracle.nlp import TargetNlp
    from oracle.ipm import IpmOptions
    p, mod = nmpc.prob, nmpc.oracle
    tn = TargetNlp(nmpc.ss, mod)
    ysp, usp, xsp = [np.asarray(v, dtype=float) for v in p.defSP(0.0)]
    for key, exp_ in KAT["KAT3"].items():
        d = np.array([0.0, float(key)])
        par = np.concatenate([usp, ysp, xsp, d, p.u0, np.zeros(4), [0.0], np.zeros(3), np.zeros(2)])
        guess = np.concatenate([p.x0_m, p.u0, mod.orc_fy(p.x0_m, p.u0, d, 0.0, np.zeros(2)).ravel()])
        r = tn.solve(guess, par, opts=IpmOptions(max_iter=100))
        assert r.status == 0
        if "xs" in exp_:
            assert np.allclose(r.x[:3], exp_["xs"], atol=2e-6) and np.allclose(r.x[3:5], exp_["us"], atol=2e-6)
        else:
            assert abs(r.x[1] - exp_["xs1"]) < 2e-6 and abs(r.x[3] - exp_["us0"]) < 2e-6


def test_unmodified_reference_example_defines_the_same_problem(nmpc):
    """Bit-exact against the stored record of the Ex_NMPC.py problem (tests/golden/problem_records.json)."""
    from problem_record import evaluate, load_records, record
    ref = load_records()["problems"]["nmpc_cstr"]
    mine = nmpc.prob
    rec = record(mine, nmpc.ss, nmpc.ocp)
    for name in ("nx", "nu", "ny", "nd", "N", "h", "Nsim", "npx", "npy"):
        assert ref[name] == rec[name]
    assert ref["flags"] == rec["flags"]
    for pt, ev_ref in zip(ref["points"], ref["evals"]):
        ev = evaluate(mine, pt)
        assert np.array_equal(ev_ref["Fx_model"], ev["Fx_model"]) and np.array_equal(ev_ref["Fx_p"], ev["Fx_p"])
    oa, ob = ref["ocp"], rec["ocp"]
    assert np.array_equal(oa["w_lb"], ob["w_lb"]) and np.array_equal(oa["w_ub"], ob["w_ub"]) and np.array_equal(oa["g_lb"], ob["g_lb"])
    assert np.array_equal(oa["g_ub"], ob["g_ub"]) and oa["off"] == ob["off"] and ref["ss"]["off"] == rec["ss"]["off"]
    assert np.array_equal(ref["ss"]["w_lb"], rec["ss"]["w_lb"]) and np.array_equal(ref["ss"]["w_ub"], rec["ss"]["w_ub"])
    for k in ("Q", "R", "P0"):
        assert np.array_equal(ref["estimator"][k], rec["estimator"][k])


@pytest.mark.skipif(not os.path.isdir(REFERENCE), reason="reference checkout not present")
@pytest.mark.parametrize("fname", ["Ex_LMPC_CSTR.py", "Ex_LMPC_WB.py", "Ex_NMPC.py", "Ex_LMPC_nlplant.py", "Ex_LMPCxp_nlplant.py", "Ex_NMPC_dis.py"])
def test_reference_examples_load_unchanged(fname):
    ns = load_example(os.path.join(REFERENCE, fname))
    prob = build_problem(ns)
    ss, ocp = make_specs(prob)
    assert ocp.nw == prob.nx * (prob.N + 1) + prob.nu * prob.N and ocp.npar == prob.npar and ss.npar == prob.npar_ss
