"""GPU parity of the FFJORD evaluator of any depth (csrc/cnf_net.cu through pnode_b200/cnfnet.py in the generic stage loop)
against the oracle, which evaluates the module the way the reference does (autograd Hutchinson trace, second-order autograd
VJP): trajectory, lambda and every parameter gradient separately, at the bars of test_gpu_cnf.py."""
import copy

import pytest
import torch
import torch.nn as nn

from oracle import OracleODEPetsc
from pnode_b200.options import Options
from _problems import rel_err
from _workloads import CNFFunc, cnf_to

pytestmark = pytest.mark.gpu

PATH = "generic+cnf-net-rhs"
TOL = {torch.float64: 1e-10, torch.float32: 1e-4}


def _inputs(B, D, T, dtype, seed=2):
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(B, D, generator=g, dtype=torch.float64)
    u0 = torch.cat((z.view(-1), torch.zeros(B, dtype=torch.float64))).to(dtype)
    gout = torch.randn(T, B * (D + 1), generator=g, dtype=torch.float64).to(dtype)
    return u0, gout


def _run(make, dev, argv, func, u0, t, gout, method, step):
    Options.clear_all()
    Options.insert_args(argv)
    f = cnf_to(copy.deepcopy(func), dev)
    ode = make()
    ode.setupTS(u0.to(dev), f, step_size=step, method=method, enable_adjoint=True)
    y0 = u0.to(dev).clone().requires_grad_(True)
    out = ode.odeint_adjoint(y0, t.to(dev))
    (out * gout.to(dev)).sum().backward()
    return out.detach(), y0.grad, [p.grad for p in f.parameters()], ode, f


def _mine(argv, func, u0, t, gout, method, step):
    from pnode import petsc_adjoint

    return _run(lambda: petsc_adjoint.ODEPetsc(), "cuda", argv, func, u0, t, gout, method, step)


def _oracle(argv, func, u0, t, gout, method, step):
    return _run(lambda: OracleODEPetsc(argv), "cpu", argv, func, u0, t, gout, method, step)


def _compare(p, o, tol):
    assert rel_err(p[0], o[0]) < tol, ("trajectory", rel_err(p[0], o[0]))
    assert rel_err(p[1], o[1]) < tol, ("lambda", rel_err(p[1], o[1]))
    assert len(p[2]) == len(o[2])
    for i, (a, b) in enumerate(zip(p[2], o[2])):
        assert a is not None and a.shape == b.shape
        assert rel_err(a, b) < tol, ("layer %d parameter %d" % (i // 5, i % 5), rel_err(a, b))


def _same(p, q):
    assert torch.equal(p[0], q[0]) and torch.equal(p[1], q[1])
    for a, b in zip(p[2], q[2]):
        assert torch.equal(a, b)


FIXED = ["-ts_adapt_type", "none"]


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("D,hidden,B", [(43, (860, 860), 1000), (8, (80,), 77), (21, (210, 210, 210), 77), (6, (60, 60), 1),
                                        (6, (60, 60), 77)],
                         ids=["miniboone", "one-layer", "three-hidden", "two-hidden-B1", "two-hidden-B77"])
def test_rk4_matches_the_oracle(dtype, D, hidden, B):
    func = CNFFunc(B, D, hidden, dtype=dtype, seed=len(hidden))
    u0, gout = _inputs(B, D, 2, dtype)
    t = torch.tensor([0.0, 1.0], dtype=torch.float64)
    o = _oracle(FIXED, func, u0, t, gout, "rk4", 0.25)
    p = _mine(FIXED, func, u0, t, gout, "rk4", 0.25)
    assert p[3].path == PATH and p[3]._loop.steps == 4
    assert p[3]._cb_ex.reused_activations == 16  # every adjoint stage read the activation set of its forward evaluation
    _compare(p, o, TOL[dtype])


@pytest.mark.parametrize("dtype,ts_tol", [(torch.float64, "1e-6"), (torch.float32, "1e-4")], ids=["f64", "f32"])
def test_dopri5_adaptive_takes_the_oracle_s_steps(dtype, ts_tol):
    B, D = 120, 8
    func = CNFFunc(B, D, (80, 80), dtype=dtype, seed=3)
    with torch.no_grad():  # stiffer dynamics: the first big step is rejected
        for prm in func.parameters():
            prm.mul_(3.0)
    u0, gout = _inputs(B, D, 3, dtype)
    t = torch.tensor([0.0, 0.4, 1.0], dtype=torch.float64)
    argv = ["-ts_rtol", ts_tol, "-ts_atol", ts_tol]
    o = _oracle(argv, func, u0, t, gout, "dopri5", 0.5)
    p = _mine(argv, func, u0, t, gout, "dopri5", 0.5)
    assert p[3].path == PATH
    lo, lp = o[3].ts.log, p[3]._loop.attempts
    if dtype == torch.float64:
        assert any(not a[2] for a in lo), "case must contain a rejected attempt"
    assert [a[2] for a in lo] == [a[2] for a in lp], "accept/reject pattern"
    for a, b in zip(lo, lp):
        assert a[1] == pytest.approx(b[1], rel=1e-8 if dtype == torch.float64 else 2e-2)
    _compare(p, o, TOL[dtype])


@pytest.mark.parametrize("method,argv,tol,t_via_f32", [
    ("bosh3", [], 1e-10, True), ("imex", FIXED, 1e-10, True),
    ("cn", FIXED + ["-ksp_rtol", "1e-13", "-snes_rtol", "1e-13"], 1e-8, True), ("bosh3", [], 1e-10, False)],
                         ids=["3bs-adaptive", "arkimex", "cn", "3bs-adaptive-t-f64"])
def test_other_schemes_fp64(method, argv, tol, t_via_f32):
    """t_via_f32=False: a module that keeps t in fp64, from a start time off the fp32 grid."""
    B, D = 40, 5
    func = CNFFunc(B, D, (37, 129), dtype=torch.float64, seed=4, t_via_f32=t_via_f32)
    u0, gout = _inputs(B, D, 3, torch.float64)
    t = torch.tensor([0.0, 0.5, 1.0], dtype=torch.float64) + (0.0 if t_via_f32 else 0.3)
    o = _oracle(argv, func, u0, t, gout, method, 0.25)
    p = _mine(argv, func, u0, t, gout, method, 0.25)
    assert p[3].path == PATH and p[3]._cb_ex.spec.t_via_f32 == int(t_via_f32)
    _compare(p, o, tol)


def test_single_time_point_fp64():
    B, D = 50, 8
    func = CNFFunc(B, D, (80, 80), dtype=torch.float64, seed=6)
    u0, gout = _inputs(B, D, 1, torch.float64)
    t = torch.tensor([0.8], dtype=torch.float64)
    argv = ["-ts_rtol", "1e-6", "-ts_atol", "1e-6"]
    o = _oracle(argv, func, u0, t, gout, "dopri5", 0.1)
    p = _mine(argv, func, u0, t, gout, "dopri5", 0.1)
    assert p[3].path == PATH and p[0].shape == (1, B * (D + 1))
    _compare(p, o, 1e-10)


def test_probe_is_sampled_like_the_generic_path_when_absent():
    """odefunc.py:359-364: `_e` is drawn inside the first evaluation of a solve; the evaluator draws the same one."""
    B, D = 32, 8
    func = cnf_to(CNFFunc(B, D, (80, 80), dtype=torch.float32), "cuda")
    u0, gout = _inputs(B, D, 2, torch.float32)
    t = torch.tensor([0.0, 1.0]).cuda()
    res = []
    for argv in ([], ["-pnode_fused", "0"]):
        from pnode import petsc_adjoint

        Options.clear_all()
        Options.insert_args(FIXED + argv)
        func.base_func.before_odeint()  # e <- None
        ode = petsc_adjoint.ODEPetsc()
        ode.setupTS(u0.cuda(), func, step_size=0.25, method="rk4")
        torch.manual_seed(77)
        out = ode.odeint_adjoint(u0.cuda(), t)
        res.append((ode.path, func.base_func._e.clone(), out.detach()))
    assert res[0][0] == PATH and res[1][0] == "generic"
    assert res[0][1].shape == (B, D) and torch.equal(res[0][1], res[1][1])
    assert rel_err(res[0][2], res[1][2]) < 1e-4


def test_num_evals_counts_like_the_generic_path():
    """ODEfunc._num_evals (FFJORD's NFE counter) advances on the device by the generic path's count: forward with
    rejected attempts, then the adjoint sweep."""
    B, D = 64, 8
    base = CNFFunc(B, D, (80,), dtype=torch.float64, seed=3)
    with torch.no_grad():
        for prm in base.parameters():
            prm.mul_(3.0)
    u0, gout = _inputs(B, D, 2, torch.float64)
    t = torch.tensor([0.0, 1.0], dtype=torch.float64).cuda()
    counts = []
    for argv in ([], ["-pnode_fused", "0"]):
        from pnode import petsc_adjoint

        Options.clear_all()
        Options.insert_args(["-ts_rtol", "1e-7", "-ts_atol", "1e-7"] + argv)
        func = cnf_to(copy.deepcopy(base), "cuda")
        ode = petsc_adjoint.ODEPetsc()
        ode.setupTS(u0.cuda(), func, step_size=0.5, method="dopri5")
        func.base_func.before_odeint(e=base.base_func._e.cuda())
        y0 = u0.cuda().clone().requires_grad_(True)
        out = ode.odeint_adjoint(y0, t)
        after_forward = float(func.base_func._num_evals)
        (out * gout.cuda()).sum().backward()
        counts.append((ode.path, after_forward, float(func.base_func._num_evals), len(ode._loop.attempts)))
    assert counts[0][0] == PATH and counts[1][0] == "generic"
    assert counts[0][1:] == counts[1][1:] and counts[0][1] > 0
    assert any(not a[2] for a in ode._loop.attempts), "case must contain a rejected attempt"


def test_kept_activation_sets_equal_re_evaluation_and_runs_repeat_bit_for_bit():
    B, D = 77, 21
    func = CNFFunc(B, D, (210, 210, 210), dtype=torch.float64, seed=8)
    u0, gout = _inputs(B, D, 3, torch.float64)
    t = torch.tensor([0.0, 0.5, 1.0], dtype=torch.float64)
    argv = ["-ts_rtol", "1e-6", "-ts_atol", "1e-6"]
    a = _mine(argv, func, u0, t, gout, "dopri5", 0.1)
    b = _mine(argv, func, u0, t, gout, "dopri5", 0.1)
    c = _mine(argv + ["-pnode_cnf_save_mb", "0"], func, u0, t, gout, "dopri5", 0.1)
    assert a[3].path == b[3].path == c[3].path == PATH
    assert a[3]._cb_ex.reused_activations > 0 and c[3]._cb_ex.reused_activations == 0
    _same(a, b)
    _same(a, c)


def test_rk4_training_step_replays_from_a_cuda_graph():
    """The whole forward + adjoint pass launches without reading the device (t reaches the gate kernel as an argument), so
    a torch.cuda.graph around the caller's step replays it on new data bit for bit."""
    from pnode import petsc_adjoint

    B, D = 200, 43
    func = cnf_to(CNFFunc(B, D, (86, 86), dtype=torch.float32, seed=2), "cuda")
    Options.clear_all()
    Options.insert_args(FIXED)
    u_static = _inputs(B, D, 2, torch.float32, seed=0)[0].cuda()
    g_static = _inputs(B, D, 2, torch.float32, seed=9)[1].cuda()
    t = torch.tensor([0.0, 1.0], dtype=torch.float64).cuda()
    ode = petsc_adjoint.ODEPetsc()
    ode.setupTS(u_static, func, step_size=0.25, method="rk4", enable_adjoint=True)

    def one_pass():
        for p in func.parameters():
            p.grad = None
        y0 = u_static.clone().requires_grad_(True)
        out = ode.odeint_adjoint(y0, t)
        (out * g_static).sum().backward()
        return out.detach(), y0.grad, [p.grad for p in func.parameters()]

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            one_pass()
    torch.cuda.current_stream().wait_stream(s)
    assert ode.path == PATH
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = one_pass()
    for seed in (1, 2):
        u_static.copy_(_inputs(B, D, 2, torch.float32, seed=seed)[0].cuda())
        graph.replay()
        torch.cuda.synchronize()
        got = (captured[0].clone(), captured[1].clone(), [g.clone() for g in captured[2]])
        want = one_pass()
        torch.cuda.synchronize()
        _same(got, want)


def test_declines():
    from pnode import petsc_adjoint

    u0, gout = _inputs(64, 6, 2, torch.float64)
    t = torch.tensor([0.0, 1.0], dtype=torch.float64)
    # the POWER shape keeps the fused sweeps
    p = _mine(["-ts_rtol", "1e-6", "-ts_atol", "1e-6"], CNFFunc(64, 6, (60,), dtype=torch.float64), u0, t, gout, "dopri5",
              0.05)
    assert p[3].path == "fused-cnf-rk"
    # -pnode_fused 0: the module path
    p = _mine(FIXED + ["-pnode_fused", "0"], CNFFunc(64, 6, (60, 60), dtype=torch.float64), u0, t, gout, "rk4", 0.25)
    assert p[3].path == "generic"
    # another nonlinearity
    func = CNFFunc(64, 6, (60, 60), dtype=torch.float64)
    func.base_func.diffeq.activation_fns[0] = nn.Tanh()
    p = _mine(FIXED, func, u0, t, gout, "rk4", 0.25)
    assert p[3].path == "generic"
    # beyond one product's reduction length (2 x batch > 65535 in fp64)
    B = 40000
    func = cnf_to(CNFFunc(B, 6, (60, 60), dtype=torch.float64), "cuda")
    Options.clear_all()
    ode = petsc_adjoint.ODEPetsc()
    ode.setupTS(_inputs(B, 6, 1, torch.float64)[0].cuda(), func, step_size=0.25, method="rk4")
    assert ode._rhs_kind == "torch"
