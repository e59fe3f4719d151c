"""Per-hidden-unit parity of the fused fp64 spiral adjoint's parameter gradient (csrc/mlp_rk.cu) against the oracle.

The adjoint spreads the 50 x 32 (unit, trajectory) pairs of a warp's stage over the lanes in three parts (units 0..31,
32..47, 48..49), with partial sums per part that are combined per unit at the end, and it accumulates the W2 gradient as
sum v - 2 sum v r (r = 1 / (e^{2z} + 1)).  A max-norm error over a whole gradient can hide one wrong unit, so every unit's
W1 row, b1 entry and W2 column is held to the bar on its own, at a large-kernel batch with a ragged last tile, with stage
checkpoints and with solution checkpoints only."""
import copy

import pytest
import torch

from oracle import OracleODEPetsc
from pnode_b200.options import Options
from _problems import SpiralFunc, spiral_inputs

pytestmark = pytest.mark.gpu
TOL = 1e-10
BATCH = 5000  # above the small-batch kernels' limit; 5000 = 39 * 128 + 8 leaves a ragged last tile
HIDDEN = 50


def _rel(a, b):
    a = a.detach().double().cpu().reshape(-1)
    b = b.detach().double().cpu().reshape(-1)
    den = float(b.norm())
    return float((a - b).norm()) / (den if den > 0 else 1.0)


def _grads(func, u0, t, gout, argv, oracle):
    if oracle:
        f = copy.deepcopy(func).double()
        ode = OracleODEPetsc(argv)
        ode.setupTS(u0.double(), f, step_size=0.025, method="rk4", enable_adjoint=True)
        y0 = u0.double().clone().requires_grad_(True)
        out = ode.odeint_adjoint(y0, t)
        (out * gout.double()).sum().backward()
        return ode, [p.grad.detach().cpu() for p in f.parameters()]
    from pnode import petsc_adjoint

    Options.clear_all()
    Options.insert_args(argv)
    f = copy.deepcopy(func).cuda()
    ode = petsc_adjoint.ODEPetsc()
    ode.setupTS(u0.cuda(), f, step_size=0.025, method="rk4", enable_adjoint=True)
    y0 = u0.cuda().clone().requires_grad_(True)
    out = ode.odeint_adjoint(y0, t.cuda())
    (out * gout.cuda()).sum().backward()
    torch.cuda.synchronize()
    return ode, [p.grad.detach().cpu() for p in f.parameters()]


@pytest.fixture(scope="module", params=[0.0, 0.2], ids=["bias0", "bias0.2"])
def spiral_mu(request):
    """(oracle gradients, {solution_only: fused gradients}) for one seeded spiral model at BATCH trajectories."""
    func = SpiralFunc(dtype=torch.float64, hidden=HIDDEN, bias_std=request.param, seed=5)
    u0, t, gout = spiral_inputs(BATCH, dtype=torch.float64, seed=7)
    argv = ["-ts_adapt_type", "none"]
    _, ref = _grads(func, u0, t, gout, argv, oracle=True)
    got = {}
    for so in (False, True):
        ode, g = _grads(func, u0, t, gout, argv + (["-ts_trajectory_solution_only", "1"] if so else []), oracle=False)
        assert ode.path == "fused-mlp-rk" and ode._fused.solution_only == so
        got[so] = g
    return ref, got


@pytest.mark.parametrize("solution_only", [False, True], ids=["stages", "solution_only"])
def test_every_hidden_unit_matches_the_oracle(spiral_mu, solution_only):
    ref, got = spiral_mu
    w1, b1, w2, b2 = got[solution_only]
    rw1, rb1, rw2, rb2 = ref
    assert w1.shape == (HIDDEN, 2) and w2.shape == (2, HIDDEN)
    bad = []
    for j in range(HIDDEN):
        for name, a, b in (("W1 row", w1[j], rw1[j]), ("b1", b1[j], rb1[j]), ("W2 column", w2[:, j], rw2[:, j])):
            e = _rel(a, b)
            if not e < TOL:
                bad.append("unit %d %s: %.3g" % (j, name, e))
    assert not bad, "; ".join(bad)
    assert _rel(b2, rb2) < TOL


def test_solution_only_gradients_are_bit_identical(spiral_mu):
    _, got = spiral_mu
    assert all(torch.equal(a, b) for a, b in zip(got[False], got[True]))
