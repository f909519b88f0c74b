"""Every example file the reference ships, through its restatement under examples/ (test_examples_equivalence.py pins
each restatement to the unmodified file): the device code (run on the CPU through the harness) must reproduce the
oracle's closed loop - same IPOPT statuses and iteration counts, trajectories to 1e-6.

Covers what the four BASELINE configurations do not: a discrete-time model with `if_else` clamps, Delta-u bounds and
a user terminal cost (Ex_NMPC_dis.py), nx != nxp (Ex_LMPCxp_nlplant.py), linear model on a nonlinear plant."""
import numpy as np
import pytest

from conftest import _bundle
from problem_record import PAIRS

RESTATED = {fname: name for name, fname, _ in PAIRS}
CASES = [("Ex_NMPC_dis.py", 6, ()), ("Ex_LMPC_nlplant.py", 8, ()), ("Ex_LMPCxp_nlplant.py", 8, ()),
         ("Ex_LMPC_CSTR.py", 6, ()), ("Ex_LMPC_WB.py", 6, ()), ("Ex_NMPC.py", 4, ())]


@pytest.mark.parametrize("fname,nsteps,edits", CASES)
def test_reference_file_closed_loop(fname, nsteps, edits):
    from harness_loop import HarnessLoop
    from oracle.closed_loop import OracleLoop
    b = _bundle(RESTATED[fname])
    p = b.prob
    ref = OracleLoop(p, b.ss, b.ocp, b.oracle).run(Nsim=nsteps)
    rec = HarnessLoop(b, 1).run(nsteps)
    assert np.array_equal(rec["STATUS_DYN"][:, 0], ref["STATUS_DYN"]) and np.array_equal(rec["ITER_DYN"][:, 0], ref["ITER_DYN"])
    assert np.array_equal(rec["STATUS_SS"][:, 0], ref["STATUS_SS"])
    for key in ("U", "X_HAT", "D_HAT", "XS", "US", "Xp", "Yp"):
        assert np.abs(rec[key][:, 0, :] - ref[key]).max() < 1e-6, key
