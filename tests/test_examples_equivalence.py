"""The problem files under examples/ are condensed restatements of the reference's Ex_*.py.  Every one of them must
define the SAME problem as the unmodified reference file: dimensions, flags, model / plant / output maps and costs
evaluated at random points, set-points, parameters, bounds, parameter offsets, estimator data and initial state.
The reference side is stored in tests/golden/problem_records.json (see tests/problem_record.py); its `source` field
says whether it was recorded from the unmodified files or from restatements that this test had checked against them.
This is what lets the tests use the oracle fixtures generated from the unmodified files (tests/golden/make_golden.py)."""
import numpy as np
import pytest

import __graft_entry__ as entry
from problem_record import PAIRS, load_records, evaluate, plain, record

REF = load_records()


def _same(a, b):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    return a.shape == b.shape and np.allclose(a, b, rtol=1e-12, atol=1e-300)


@pytest.mark.parametrize("name,fname,edits", PAIRS)
def test_example_restates_the_reference_file(name, fname, edits):
    ref = REF["problems"][name]
    mine, ss_b, ocp_b = entry._problem(name)
    rec = record(mine, ss_b, ocp_b)
    for attr in ("nx", "nxp", "nu", "ny", "nd", "N", "h", "npx", "npy", "npxp", "npyp", "nxi"):
        assert ref[attr] == rec[attr], attr
    assert ref["flags"] == rec["flags"]
    for attr in ("x0_p", "x0_m", "u0", "dhat0"):
        assert _same(ref[attr], rec[attr]), attr
    for pt, ev_ref in zip(ref["points"], ref["evals"]):        # the maps of both problems at the same points
        ev = evaluate(mine, pt)
        for fn, val in ev_ref.items():
            assert _same(val, ev[fn]), fn
    assert (ref["defSP"] is None) == (rec["defSP"] is None)
    if rec["defSP"] is not None:
        for t, a, b in zip(REF["times"], ref["defSP"], rec["defSP"]):
            assert len(a) == len(b) and all(_same(u, v) for u, v in zip(a, b)), ("defSP", t)
    assert sorted(ref["params"]) == sorted(rec["params"])
    for fn in rec["params"]:
        for t, a, b in zip(REF["times"], ref["params"][fn], rec["params"][fn]):
            assert _same(a, b), (fn, t)
    for tag in ("ocp", "ss"):
        for k in ("w_lb", "w_ub", "g_lb", "g_ub"):
            assert np.array_equal(ref[tag][k], rec[tag][k]), (tag, k)
        assert ref[tag]["off"] == rec[tag]["off"], tag
    for k in ("flags", "yFree", "DuFree", "uses_uprev"):
        assert ref["ocp"][k] == rec["ocp"][k], k
    ea, eb = ref["estimator"], rec["estimator"]
    assert ea["type"] == eb["type"]
    for k in ("Q", "R", "K", "P0", "dmin", "dmax"):
        assert (ea[k] is None) == (eb[k] is None), k
        if eb[k] is not None:
            assert _same(ea[k], eb[k]), k
    assert ref["sol_optss"] == plain(mine.sol_optss) and ref["sol_optdyn"] == plain(mine.sol_optdyn)
    assert (ref["R_wn"] is None) == (rec["R_wn"] is None) and (rec["R_wn"] is None or _same(ref["R_wn"], rec["R_wn"]))
