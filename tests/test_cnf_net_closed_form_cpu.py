"""The closed form csrc/cnf_net.cu evaluates (tests/_cnf_net_model.py) against torch autograd through the FFJORD module
itself (_workloads.CNFFunc: autograd Hutchinson trace, and a second backward for the adjoint), in fp64 on the CPU: the
right-hand side F, J^T w and the five gradients of every layer, for networks of one to four layers, ragged widths, units
above the softplus threshold and both ways a module may round t."""
import pytest
import torch

import _cnf_net_model as model
from _workloads import CNFFunc


def _case(B, D, hidden, seed, via_f32=True, saturate=0):
    func = CNFFunc(B, D, hidden, dtype=torch.float64, seed=seed, t_via_f32=via_f32)
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


def _autograd(func, u, w, t):
    y = u.clone().requires_grad_(True)
    out = func(t, y)
    params = list(func.parameters())
    g = torch.autograd.grad(out, [y] + params, w)
    return out.detach(), g[0], list(g[1:])


def _rel(a, b):
    a, b = a.detach(), b.detach()
    den = float(b.norm())
    return float((a - b).norm()) / (den if den > 0 else 1.0)


def _tau(t, via_f32):
    return float(torch.tensor(t, dtype=torch.float32)) if via_f32 else t


@pytest.mark.parametrize("D,hidden", [(6, ()), (6, (60,)), (5, (37, 129)), (43, (86, 86)), (7, (16, 24, 16))],
                         ids=["L1", "L2", "L3-ragged", "L3-miniboone-like", "L4"])
@pytest.mark.parametrize("via_f32", [True, False], ids=["t-f32", "t-f64"])
def test_closed_form_matches_autograd(D, hidden, via_f32):
    B, t = 9, 0.37
    func, layers, u, w = _case(B, D, hidden, seed=len(hidden) + D, via_f32=via_f32)
    F_ref, jtw_ref, gp_ref = _autograd(func, u, w, t)
    e = func.base_func._e
    tau = _tau(t, via_f32)
    F, cache = model.forward(layers, u[:B * D].view(B, D), e, tau)
    jtw, grads = model.vjp(layers, cache, e, w, tau)
    assert _rel(F, F_ref) < 1e-12
    assert _rel(jtw, jtw_ref) < 1e-12
    assert float(jtw[B * D:].detach().abs().max()) == 0.0 and float(jtw_ref[B * D:].abs().max()) == 0.0
    flat = [g for per_layer in grads for g in per_layer]
    assert len(flat) == len(gp_ref) == 5 * (len(hidden) + 1)
    for i, (a, b) in enumerate(zip(flat, gp_ref)):
        assert a.shape == b.shape, i
        assert _rel(a, b) < 1e-12, ("layer %d parameter %d" % (i // 5, i % 5), _rel(a, b))


def test_time_rounding_is_visible():
    """The model evaluated with the wrong rounding of t is off by far more than the 1e-12 bar: the cases above pin it."""
    B, D, t = 9, 6, 0.37
    func, layers, u, w = _case(B, D, (60,), seed=3, via_f32=True)
    F_ref = _autograd(func, u, w, t)[0]
    F_wrong = model.forward(layers, u[:B * D].view(B, D), func.base_func._e, t)[0]
    assert _rel(F_wrong, F_ref) > 1e-10


@pytest.mark.parametrize("hidden", [(60,), (37, 129)])
def test_softplus_threshold(hidden):
    """Units above torch's softplus threshold (a > 20): derivative exactly 1, second derivative exactly 0.  sigmoid(20) is
    1 - 2e-9, so a model without the threshold misses the fp64 bar."""
    B, D, t = 9, 5, 0.61
    func, layers, u, w = _case(B, D, hidden, seed=11, saturate=4)
    F_ref, jtw_ref, gp_ref = _autograd(func, u, w, t)
    e, tau = func.base_func._e, _tau(t, True)
    F, cache = model.forward(layers, u[:B * D].view(B, D), e, tau)
    a0 = cache[0]["gam"] * cache[0]["P"] + model.gates(layers, tau)[0][1]
    assert bool((a0[:, :4] > 20).all()) and bool((a0[:, :4] < 22).all()) and bool((a0[:, 4:] < 20).all())
    jtw, grads = model.vjp(layers, cache, e, w, tau)
    assert _rel(F, F_ref) < 1e-12 and _rel(jtw, jtw_ref) < 1e-12
    for a, b in zip([g for gl in grads for g in gl], gp_ref):
        assert _rel(a, b) < 1e-12

    # the same closed form with the plain sigmoid in place of the thresholded derivative
    plain = model._softplus_sigmoid
    try:
        model._softplus_sigmoid = lambda a: (torch.nn.functional.softplus(a), torch.sigmoid(a))
        F2, cache2 = model.forward(layers, u[:B * D].view(B, D), e, tau)
        jtw2, grads2 = model.vjp(layers, cache2, e, w, tau)
    finally:
        model._softplus_sigmoid = plain
    # the bias gradient of the saturated units goes through their softplus slope alone
    assert _rel(grads[0][1][:4], gp_ref[1][:4]) < 1e-12
    assert _rel(grads2[0][1][:4], gp_ref[1][:4]) > 1e-10


@pytest.mark.parametrize("hidden", [(), (60,), (37, 129), (16, 24, 16)])
def test_recogniser_probe_formula(hidden):
    """fused.cnf_closed_form (the numerical probe of the recogniser) is the same forward as the host model."""
    from pnode_b200.fused import cnf_closed_form

    B, D = 9, 5
    func, layers, u, _ = _case(B, D, hidden, seed=5)
    z, e = u[:B * D].view(B, D), func.base_func._e
    t = torch.tensor(0.3).to(torch.float64)
    with torch.no_grad():
        f, div = cnf_closed_form(layers, z, e, t)
        F = model.forward(layers, z, e, float(t))[0]
    assert _rel(torch.cat((f.reshape(-1), -div)), F) < 1e-13


def test_descriptor_layout_and_sizes(tmp_path):
    """pnode_cnfnet_desc as a C compiler lays it out equals its ctypes mirror, and the host half of csrc/cnf_net.cu (no
    kernel launched) sizes the buffers and declines what one sliced product cannot take."""
    import ctypes as C
    import os
    import subprocess

    from pnode_b200 import _lib
    from pnode_b200.cnfnet import CnfNetCallbacks, _desc_for
    from pnode_b200.fused import CnfSpec

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "desc.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "pnode_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu %zu\\n", sizeof(pnode_cnfnet_desc), '
                   'offsetof(pnode_cnfnet_desc, d_weight), offsetof(pnode_cnfnet_desc, d_gate_bias), '
                   'offsetof(pnode_cnfnet_desc, mu_hgb_off), offsetof(pnode_cnfnet_desc, d_e)); return 0; }\n')
    exe = tmp_path / "desc"
    subprocess.run(["gcc", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    d = _lib.CnfNetDesc
    assert got == [C.sizeof(d), d.d_weight.offset, d.d_gate_bias.offset, d.mu_hgb_off.offset, d.d_e.offset]

    lib = _lib.load()

    def spec(B, D, hidden):
        func = CNFFunc(B, D, hidden, dtype=torch.float64)
        return CnfSpec(func.base_func, func.base_func.diffeq.layers, B, D)

    s = spec(1000, 43, (860, 860))
    for dtype in (torch.float64, torch.float32):
        d = _desc_for(s, dtype)
        assert CnfNetCallbacks.supported(s, dtype)
        esz = 8 if dtype == torch.float64 else 4
        pq = 2 * 1000 * (860 + 860 + 43) * esz  # [P; Q] of every layer
        assert pq < lib.pnode_cnfnet_act_bytes(C.byref(d)) < pq + 64 * 2000 * (43 + 860 + 860) + (1 << 20)
        assert lib.pnode_cnfnet_work_bytes(C.byref(d)) > 0 and lib.pnode_cnfnet_weight_bytes(C.byref(d)) > 0
    big = spec(32768, 6, (60, 60))  # 2B = 65536 rows: one past the fp64 (I8X) reduction limit, within TF32's
    assert not CnfNetCallbacks.supported(big, torch.float64) and b"reduction length" in lib.pnode_last_error()
    assert CnfNetCallbacks.supported(big, torch.float32)
    assert CnfNetCallbacks.supported(spec(32767, 6, (60, 60)), torch.float64)
    assert not CnfNetCallbacks.supported(spec(10, 6, (8,) * 8), torch.float64)  # 9 layers
