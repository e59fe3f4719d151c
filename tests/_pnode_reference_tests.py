"""The original pnode project's tests/test_pnode.py, restated in its own style: a script that hands PETSc its options with
`petsc4py.init`, imports `petsc_adjoint` from `pnode` and solves the ROBER problem with `ODEPetsc().setupTS(...)` and
`odeint_adjoint`, asserting that project's known answers.  It goes through the drop-in packages `pnode` and `petsc4py` of
this repository exactly as a script written for the original does.  Not collected by pytest on its own (the options of a
module-level `petsc4py.init` would be cleared between tests): tests/test_reference_suite_cpu.py loads it afresh per test.
ROBER fixture (rate constants, output times, per-step step sizes, SciPy BDF ground truth): tests/_problems.py."""
import sys

import numpy as np
import petsc4py
import pytest
import torch

petsc4py.init(sys.argv + ["-ts_adapt_type", "none", "-ts_trajectory_type", "memory"])

from petsc4py import PETSc  # noqa: E402
from pnode import petsc_adjoint  # noqa: E402
from _problems import ROBER_STEPS, ROBER_T, Rober, RoberEX, RoberIM, rober_truth  # noqa: E402


def _solve(funcs, **kw):
    true_y = rober_truth()
    true_y0 = true_y[0]
    ode = petsc_adjoint.ODEPetsc()
    if len(funcs) == 2:
        kw["func2"] = funcs[1]
    ode.setupTS(true_y0, funcs[0], step_size=ROBER_STEPS, enable_adjoint=True, **kw)
    pred_y = ode.odeint_adjoint(true_y0, ROBER_T)
    loss = torch.mean(torch.abs(pred_y - true_y))
    std = torch.std(torch.abs(pred_y - true_y))
    loss.backward()
    return loss.item(), std.item()


def test_petsc_scalartype():
    assert PETSc.ScalarType == np.float64


def test_petsc_implicit_odesolver():
    loss, std = _solve([Rober()], method="cn", implicit_form=True)
    assert loss == pytest.approx(1.85e-6, abs=1e-6)
    assert std == pytest.approx(3.36e-6, abs=1e-6)


def test_petsc_imex_odesolver():
    loss, std = _solve([RoberIM(), RoberEX()], method="imex", implicit_form=True, imex_form=True)
    assert loss == pytest.approx(3.11e-6, abs=3e-6)
    assert std == pytest.approx(5.65e-6, abs=3e-6)


def test_petsc_explicit_odesolver():
    loss, std = _solve([Rober()], method="rk3")
    assert loss == pytest.approx(1.85e-6, abs=1e-6)
    assert std == pytest.approx(3.21e-6, abs=1e-6)
