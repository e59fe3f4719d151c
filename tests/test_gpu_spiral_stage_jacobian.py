"""The stage Jacobians the fp64 spiral forward sweep keeps next to its stage values (csrc/mlp_rk.cu StageJac) and which the
adjoint sweep uses for the stage VJP: each stored J_i must be df/dy of the right-hand side at the stored Y_i."""
import ctypes

import pytest
import torch

from _problems import SpiralFunc, rel_err
from pnode_b200 import _lib, tableaux
from pnode_b200.fused import FusedMlpRK, _tableau_struct, recognise_mlp


def _rows(dim, hidden, dtype, stages=4):
    desc = _lib.MlpDesc()
    desc.dim, desc.hidden, desc.phi, desc.dtype = dim, hidden, 1, dtype
    tab = _tableau_struct(tableaux.RK["5dp" if stages == 7 else "4"])
    return _lib.load().pnode_mlp_rk_ckpt_rows(ctypes.byref(desc), ctypes.byref(tab))


def test_checkpoint_rows_per_stage():
    """Y_i and, in the fp64 sweeps of the 50-unit shapes with one or two state components, J_i row-major; Y_i alone
    elsewhere."""
    assert _rows(2, 50, _lib.F64) == 6 and _rows(2, 50, _lib.F64, stages=7) == 6
    assert _rows(1, 50, _lib.F64) == 2 and _rows(3, 50, _lib.F64) == 3 and _rows(4, 50, _lib.F64) == 4
    assert _rows(2, 50, _lib.F32) == 2 and _rows(2, 100, _lib.F64) == 2 and _rows(4, 50, _lib.F32) == 4


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["4", "5dp"], ids=["rk4", "fixed_dopri5"])
def test_stored_stage_jacobians_match_autograd(method):
    dev = torch.device("cuda:0")
    n = 5000  # above the small-batch kernels' limit: the large-batch sweep writes the Jacobian rows
    func = SpiralFunc().to(dev)
    g = torch.Generator().manual_seed(1)
    u0 = ((torch.rand(n, 1, 2, generator=g, dtype=torch.float64) * 2 - 1) * 2).to(dev)
    fused = FusedMlpRK(recognise_mlp(func, u0), tableaux.RK[method], torch.float64, dev)
    times = [0.025 * i for i in range(10)]
    _, ckpt, (_, nsteps, _) = fused.forward(u0.reshape(-1), times, 0.025, True)
    torch.cuda.synchronize()
    s = tableaux.RK[method].s
    assert tuple(ckpt.shape) == (nsteps, s, 6, n)
    for step in range(nsteps):
        for i in range(s):
            y = ckpt[step, i, :2].t().contiguous()                         # [n, 2]
            got = ckpt[step, i, 2:].view(2, 2, n).permute(2, 0, 1)         # [n, d, e] = df_d / dy_e
            # trajectories are independent: d/dy of sum_b f(y_b) is the per-trajectory Jacobian, [d, b, e]
            ref = torch.autograd.functional.jacobian(lambda yy: func(None, yy).sum(0), y).permute(1, 0, 2)
            assert rel_err(got, ref) < 1e-13, (step, i, rel_err(got, ref))
