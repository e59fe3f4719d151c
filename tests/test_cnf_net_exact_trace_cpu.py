"""The exact trace (divergence_bf) of the FFJORD evaluator of any depth: the closed form csrc/cnf_net.cu evaluates with D
tangent chains (tests/_cnf_exact.py) against torch autograd through the module itself (D autograd calls per evaluation, a
second backward for the adjoint), in fp64 on the CPU -- F, J^T w and the five gradients of every layer, for one to four
layers, both ways a module may round t and units above the softplus threshold -- and the host half of the evaluator: the
descriptor field that selects the trace, and the (D + 1) B row limit."""
import ctypes as C
import os
import subprocess

import pytest
import torch

import _cnf_exact as xmodel


def _autograd(func, u, w, t):
    y = u.clone().requires_grad_(True)
    out = func(t, y)
    g = torch.autograd.grad(out, [y] + list(func.parameters()), w)
    return out.detach(), g[0], list(g[1:])


def _rel(a, b):
    a, b = a.detach(), b.detach()
    den = float(b.norm())
    return float((a - b).norm()) / (den if den > 0 else 1.0)


def _tau(t, via_f32):
    return float(torch.tensor(t, dtype=torch.float32)) if via_f32 else t


def _case(B, D, hidden, seed, via_f32=True, saturate=0):
    func = xmodel.exact_cnf(B, D, hidden, dtype=torch.float64, seed=seed, t_via_f32=via_f32)
    layers = list(func.base_func.diffeq.layers)
    if saturate:
        with torch.no_grad():  # push the first units of the first layer just past the softplus threshold (a ~ 21)
            layers[0]._layer.bias[:saturate] = 42.4
            layers[0]._layer.weight[:saturate] *= 0.1
            layers[0]._hyper_gate.weight[:saturate] = 0.0
            layers[0]._hyper_gate.bias[:saturate] = 0.0
            layers[0]._hyper_bias.weight[:saturate] = 0.0
    g = torch.Generator().manual_seed(seed + 7)
    u = torch.cat((torch.randn(B * D, generator=g, dtype=torch.float64), torch.randn(B, generator=g, dtype=torch.float64)))
    w = torch.randn(B * (D + 1), generator=g, dtype=torch.float64)
    return func, layers, u, w


def _check(func, layers, u, w, t, tau, B, D):
    F_ref, jtw_ref, gp_ref = _autograd(func, u, w, t)
    F, cache = xmodel.forward(layers, u[:B * D].view(B, D), tau)
    jtw, grads = xmodel.vjp(layers, cache, w, tau)
    assert _rel(F, F_ref) < 1e-12, _rel(F, F_ref)
    assert _rel(jtw, jtw_ref) < 1e-12, _rel(jtw, jtw_ref)
    assert float(jtw[B * D:].detach().abs().max()) == 0.0 and float(jtw_ref[B * D:].abs().max()) == 0.0
    flat = [g for per_layer in grads for g in per_layer]
    assert len(flat) == len(gp_ref) == 5 * len(layers)
    for i, (a, b) in enumerate(zip(flat, gp_ref)):
        assert a.shape == b.shape, i
        assert _rel(a, b) < 1e-12, ("layer %d parameter %d" % (i // 5, i % 5), _rel(a, b))
    return F, F_ref


@pytest.mark.parametrize("D,hidden", [(6, ()), (6, (60,)), (5, (37, 129)), (2, (64, 64, 64)), (7, (16, 24, 16))],
                         ids=["L1", "L2", "L3-ragged", "L4-D2", "L4"])
@pytest.mark.parametrize("via_f32", [True, False], ids=["t-f32", "t-f64"])
def test_exact_closed_form_matches_autograd(D, hidden, via_f32):
    B, t = 9, 0.37
    func, layers, u, w = _case(B, D, hidden, seed=len(hidden) + D, via_f32=via_f32)
    F, _ = _check(func, layers, u, w, t, _tau(t, via_f32), B, D)
    # the exact trace is not the Hutchinson estimate of the same network
    from _cnf_net_model import forward as hutchinson_forward

    F_h = hutchinson_forward(layers, u[:B * D].view(B, D), func.base_func._e, _tau(t, via_f32))[0]
    assert _rel(F_h[B * D:], F[B * D:]) > 1e-3


@pytest.mark.parametrize("hidden", [(60,), (37, 129)])
def test_exact_softplus_threshold(hidden):
    """Units above torch's softplus threshold (a > 20): slope exactly 1, second derivative exactly 0, in every chain."""
    B, D, t = 9, 5, 0.61
    func, layers, u, w = _case(B, D, hidden, seed=11, saturate=4)
    tau = _tau(t, True)
    _, cache = xmodel.forward(layers, u[:B * D].view(B, D), tau)
    from _cnf_net_model import gates

    a0 = cache[0]["gam"] * cache[0]["P"] + gates(layers, tau)[0][1]
    assert bool((a0[:, :4] > 20).all()) and bool((a0[:, :4] < 22).all()) and bool((a0[:, 4:] < 20).all())
    _check(func, layers, u, w, t, tau, B, D)


def test_eval_branch_module_takes_the_exact_trace():
    """The restated FFJORD eval-mode branch: Hutchinson in training mode, the exact trace in eval mode (D = 2)."""
    from _cnf_net_model import forward as hutchinson_forward

    B, t = 9, 0.37
    func = xmodel.eval_branch_cnf(B, (16, 16), seed=3)
    layers = list(func.base_func.diffeq.layers)
    u = torch.randn(B * 3, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    w = torch.randn(B * 3, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    tau = _tau(t, True)
    func.eval()
    _check(func, layers, u, w, t, tau, B, 2)
    func.train()
    F_ref = _autograd(func, u, w, t)[0]
    assert _rel(hutchinson_forward(layers, u[:B * 2].view(B, 2), func.base_func._e, tau)[0], F_ref) < 1e-12


@pytest.mark.parametrize("hidden", [(), (60,), (37, 129), (16, 24, 16)])
def test_recogniser_probe_formula_exact(hidden):
    """fused.cnf_closed_form(exact=True) (the recogniser's probe of the exact trace) is the host model's forward."""
    from pnode_b200.fused import cnf_closed_form

    B, D = 9, 5
    func, layers, u, _ = _case(B, D, hidden, seed=5)
    z = u[:B * D].view(B, D)
    t = torch.tensor(0.3).to(torch.float64)
    with torch.no_grad():
        f, div = cnf_closed_form(layers, z, None, t, exact=True)
        F = xmodel.forward(layers, z, float(t))[0]
    assert _rel(torch.cat((f.reshape(-1), -div)), F) < 1e-13


def _spec(B, D, hidden, trace):
    from pnode_b200.fused import CnfSpec

    func = xmodel.exact_cnf(B, D, hidden, dtype=torch.float64)
    s = CnfSpec(func.base_func, func.base_func.diffeq.layers, B, D)
    s.trace = trace
    return s


def test_descriptor_trace_field(tmp_path):
    """pnode_cnfnet_desc.trace as a C compiler lays it out equals its ctypes mirror; the fields before it keep their
    offsets; _desc_for sets it from the spec."""
    from pnode_b200 import _lib
    from pnode_b200.cnfnet import _desc_for

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "desc.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "pnode_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu\\n", sizeof(pnode_cnfnet_desc), '
                   'offsetof(pnode_cnfnet_desc, mu_hgb_off), offsetof(pnode_cnfnet_desc, d_e), '
                   'offsetof(pnode_cnfnet_desc, trace)); return 0; }\n')
    exe = tmp_path / "desc"
    subprocess.run(["gcc", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    d = _lib.CnfNetDesc
    assert got == [C.sizeof(d), d.mu_hgb_off.offset, d.d_e.offset, d.trace.offset]
    assert d.trace.offset == d.d_e.offset + 8
    assert _desc_for(_spec(4, 6, (60,), "exact"), torch.float64).trace == 1
    assert _desc_for(_spec(4, 6, (60,), "hutchinson"), torch.float64).trace == 0


def test_row_limit_and_activation_set_size():
    """(D + 1) B rows must fit one product's reduction length: 65535 in fp64 (I8X), 65536 in fp32 (TF32).  The activation
    set grows by about (D + 1) / 2 over the Hutchinson trace's."""
    from pnode_b200 import _lib
    from pnode_b200.cnfnet import CnfNetCallbacks, _desc_for
    from pnode_b200.fused import FusedCnfRK
    from pnode_b200 import tableaux

    lib = _lib.load()
    # fp64: 5 x 13107 = 65535 (at the limit), one sample more is past it; the Hutchinson trace takes both (2B rows)
    assert CnfNetCallbacks.supported(_spec(13107, 4, (60, 60), "exact"), torch.float64)
    assert not CnfNetCallbacks.supported(_spec(13108, 4, (60, 60), "exact"), torch.float64)
    assert b"reduction length" in lib.pnode_last_error()
    assert CnfNetCallbacks.supported(_spec(13108, 4, (60, 60), "hutchinson"), torch.float64)
    # fp32: 4 x 16384 = 65536
    assert CnfNetCallbacks.supported(_spec(16384, 3, (60,), "exact"), torch.float32)
    assert not CnfNetCallbacks.supported(_spec(16385, 3, (60,), "exact"), torch.float32)
    assert b"reduction length" in lib.pnode_last_error()

    D = 43
    ex, hu = _spec(1000, D, (860, 860), "exact"), _spec(1000, D, (860, 860), "hutchinson")
    for dtype in (torch.float64, torch.float32):
        a_ex = lib.pnode_cnfnet_act_bytes(C.byref(_desc_for(ex, dtype)))
        a_hu = lib.pnode_cnfnet_act_bytes(C.byref(_desc_for(hu, dtype)))
        # fp64: 44000 rows take the wider I8X slicing where the Hutchinson trace's 2000 take I8
        assert 0.9 * (D + 1) / 2 < a_ex / a_hu < 1.2 * (D + 1) / 2
        esz = 8 if dtype == torch.float64 else 4
        assert a_ex > (D + 1) * 1000 * (860 + 860 + D) * esz  # [P; Q^(0); ...] of every layer
        assert lib.pnode_cnfnet_work_bytes(C.byref(_desc_for(ex, dtype))) > 0

    # the fused two-layer sweeps carry the Hutchinson trace only
    rk4 = tableaux.lookup("rk", "4")
    assert not FusedCnfRK.supported(_spec(64, 6, (60,), "exact"), rk4, torch.float64)
