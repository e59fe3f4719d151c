"""GPU parity of the exact trace (divergence_bf) on the FFJORD evaluator of any depth (csrc/cnf_net.cu with D tangent
chains) against the oracle, which evaluates the module the way the reference does (D autograd calls per evaluation,
second-order autograd VJP): trajectory, lambda and every parameter gradient separately.  Also the module's eval-mode
branch to the exact trace, the probe's RNG draw, FFJORD's evaluation counter, kept activation sets, CUDA-graph replay
and the row limit."""
import copy

import pytest
import torch

from oracle import OracleODEPetsc
from pnode_b200.options import Options
from _cnf_exact import eval_branch_cnf, exact_cnf
from _problems import rel_err
from _workloads import CNFFunc, cnf_to

pytestmark = pytest.mark.gpu

PATH = "generic+cnf-net-rhs"
TOL = {torch.float64: 1e-10, torch.float32: 1e-4}
FIXED = ["-ts_adapt_type", "none"]


def _inputs(B, D, T, dtype, seed=2):
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(B, D, generator=g, dtype=torch.float64)
    u0 = torch.cat((z.view(-1), torch.zeros(B, dtype=torch.float64))).to(dtype)
    gout = torch.randn(T, B * (D + 1), generator=g, dtype=torch.float64).to(dtype)
    return u0, gout


def _solve(ode, f, u0, t, gout, dev):
    for p in f.parameters():
        p.grad = None
    y0 = u0.to(dev).clone().requires_grad_(True)
    out = ode.odeint_adjoint(y0, t.to(dev))
    (out * gout.to(dev)).sum().backward()
    return out.detach(), y0.grad, [p.grad for p in f.parameters()]


def _run(make, dev, argv, func, u0, t, gout, method, step):
    Options.clear_all()
    Options.insert_args(argv)
    f = cnf_to(copy.deepcopy(func), dev)
    ode = make()
    ode.setupTS(u0.to(dev), f, step_size=step, method=method, enable_adjoint=True)
    return _solve(ode, f, u0, t, gout, dev) + (ode, f)


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


def _exact(ode):
    return ode.path == PATH and ode._cb_ex.spec.trace == "exact"


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("D,hidden,B", [(2, (64, 64, 64), 100), (6, (60,), 64), (6, (60, 60), 64), (43, (86, 86), 12),
                                        (6, (60, 60), 1)],
                         ids=["D2-three-hidden", "power-one-hidden", "power-two-hidden", "miniboone-like", "B1"])
def test_rk4_matches_the_oracle(dtype, D, hidden, B):
    func = exact_cnf(B, D, hidden, dtype=dtype, seed=len(hidden) + D)
    u0, gout = _inputs(B, D, 2, dtype)
    t = torch.tensor([0.0, 1.0], dtype=torch.float64)
    o = _oracle(FIXED, func, u0, t, gout, "rk4", 0.25)
    p = _mine(FIXED, func, u0, t, gout, "rk4", 0.25)
    assert _exact(p[3]) and p[3]._loop.steps == 4
    assert p[3]._cb_ex.reused_activations == 16
    _compare(p, o, TOL[dtype])


def _to_f64(func):
    f = copy.deepcopy(func).to(torch.float64)
    f.base_func._e = f.base_func._e.to(torch.float64)
    f.y0 = tuple(x.to(torch.float64) for x in f.y0)
    return f


def test_miniboone_fp32_at_full_batch_matches_the_fp64_module_path():
    """D = 43, hidden 860-860, B = 1000 in fp32: 44000 stacked rows.  The weight gradients reduce over them in split-K slices
    of about B rows, added in order in double, so every output stays within the fp32 bar of the module path run in fp64
    (a single fp32 accumulation over all rows puts the middle layer's weight gradient 3e-4 off), and mu repeats bit for bit."""
    B, D = 1000, 43
    func = exact_cnf(B, D, (860, 860), dtype=torch.float32, seed=1)
    u0, gout = _inputs(B, D, 2, torch.float32)
    t = torch.tensor([0.0, 1.0], dtype=torch.float64)
    ref = _mine(FIXED + ["-pnode_fused", "0"], _to_f64(func), u0.double(), t, gout.double(), "rk4", 0.25)
    assert ref[3].path == "generic"
    p = _mine(FIXED, func, u0, t, gout, "rk4", 0.25)
    q = _mine(FIXED, func, u0, t, gout, "rk4", 0.25)
    assert _exact(p[3]) and p[3]._cb_ex.reused_activations == 16
    _compare(p, ref, 1e-4)
    _same(p, q)


def test_fp64_past_the_int8_row_limit_matches_the_oracle():
    """(D + 1) B = 16800 stacked rows in fp64: past PNODE_I8_MAX_K, so every product of the evaluator takes the I8X digits."""
    B, D = 2400, 6
    func = exact_cnf(B, D, (60, 60), dtype=torch.float64, seed=7)
    u0, gout = _inputs(B, D, 2, torch.float64)
    t = torch.tensor([0.0, 1.0], dtype=torch.float64)
    o = _oracle(FIXED, func, u0, t, gout, "rk4", 0.25)
    p = _mine(FIXED, func, u0, t, gout, "rk4", 0.25)
    assert _exact(p[3]) and (D + 1) * B > 16384
    _compare(p, o, 1e-10)


@pytest.mark.parametrize("dtype,ts_tol", [(torch.float64, "1e-6"), (torch.float32, "1e-4")], ids=["f64", "f32"])
def test_dopri5_adaptive_takes_the_oracle_s_steps(dtype, ts_tol):
    B, D = 60, 6
    func = exact_cnf(B, D, (60, 60), dtype=dtype, seed=3)
    with torch.no_grad():  # stiffer dynamics: the first big step is rejected
        for prm in func.parameters():
            prm.mul_(3.0)
    u0, gout = _inputs(B, D, 3, dtype)
    t = torch.tensor([0.0, 0.4, 1.0], dtype=torch.float64)
    argv = ["-ts_rtol", ts_tol, "-ts_atol", ts_tol]
    o = _oracle(argv, func, u0, t, gout, "dopri5", 0.5)
    p = _mine(argv, func, u0, t, gout, "dopri5", 0.5)
    assert _exact(p[3])
    lo, lp = o[3].ts.log, p[3]._loop.attempts
    if dtype == torch.float64:
        assert any(not a[2] for a in lo), "case must contain a rejected attempt"
    assert [a[2] for a in lo] == [a[2] for a in lp], "accept/reject pattern"
    for a, b in zip(lo, lp):
        assert a[1] == pytest.approx(b[1], rel=1e-8 if dtype == torch.float64 else 2e-2)
    _compare(p, o, TOL[dtype])


def test_bosh3_with_t_in_fp64():
    """A module that keeps t in fp64, from a start time off the fp32 grid."""
    B, D = 40, 5
    func = exact_cnf(B, D, (37, 129), dtype=torch.float64, seed=4, t_via_f32=False)
    u0, gout = _inputs(B, D, 3, torch.float64)
    t = torch.tensor([0.3, 0.8, 1.3], dtype=torch.float64)
    o = _oracle([], func, u0, t, gout, "bosh3", 0.25)
    p = _mine([], func, u0, t, gout, "bosh3", 0.25)
    assert _exact(p[3]) and p[3]._cb_ex.spec.t_via_f32 == 0
    _compare(p, o, 1e-10)


def test_eval_mode_branch_train_eval_train_on_one_solver():
    """FFJORD's ODEfunc takes the exact trace in eval mode for 2-D states whatever its divergence_fn: the verdict follows
    the module's mode across solves on one ODEPetsc, and each solve matches the oracle in that mode."""
    from pnode import petsc_adjoint

    B = 50
    base = eval_branch_cnf(B, (64, 64, 64), seed=5)
    u0, gout = _inputs(B, 2, 2, torch.float64)
    t = torch.tensor([0.0, 1.0], dtype=torch.float64)
    Options.clear_all()
    Options.insert_args(FIXED)
    f = cnf_to(copy.deepcopy(base), "cuda")
    ode = petsc_adjoint.ODEPetsc()
    for training, trace in ((True, "hutchinson"), (False, "exact"), (True, "hutchinson")):
        f.train(training)
        ref = copy.deepcopy(base).train(training)
        Options.clear_all()
        Options.insert_args(FIXED)
        ode.setupTS(u0.cuda(), f, step_size=0.25, method="rk4", enable_adjoint=True)
        p = _solve(ode, f, u0, t, gout, "cuda")
        assert ode.path == PATH and ode._cb_ex.spec.trace == trace, (training, ode.path)
        o = _oracle(FIXED, ref, u0, t, gout, "rk4", 0.25)
        _compare(p, o, 1e-10)


def test_probe_and_rng_stream_follow_the_module_path():
    """The module draws `_e` before it picks a divergence: the evaluator draws the same one for the exact trace (which does
    not read it), so `_e` and the caller's next random numbers equal the module path's."""
    from pnode import petsc_adjoint

    B, D = 32, 6
    func = cnf_to(exact_cnf(B, D, (60, 60), dtype=torch.float32), "cuda")
    u0, gout = _inputs(B, D, 2, torch.float32)
    t = torch.tensor([0.0, 1.0]).cuda()
    res = []
    for argv in ([], ["-pnode_fused", "0"]):
        Options.clear_all()
        Options.insert_args(FIXED + argv)
        func.base_func.before_odeint()  # e <- None
        ode = petsc_adjoint.ODEPetsc()
        ode.setupTS(u0.cuda(), func, step_size=0.25, method="rk4")
        torch.manual_seed(77)
        y0 = u0.cuda().clone().requires_grad_(True)
        out = ode.odeint_adjoint(y0, t)
        (out * gout.cuda()).sum().backward()
        nxt = torch.randn(8, device="cuda")
        res.append((ode.path, func.base_func._e.clone(), nxt, out.detach()))
    assert res[0][0] == PATH and res[1][0] == "generic"
    assert res[0][1].shape == (B, D) and torch.equal(res[0][1], res[1][1])
    assert torch.equal(res[0][2], res[1][2])
    assert rel_err(res[0][3], res[1][3]) < 1e-4


def test_num_evals_counts_like_the_module_path():
    B, D = 48, 6
    base = exact_cnf(B, D, (60,), dtype=torch.float64, seed=3)
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
    B, D = 40, 9
    func = exact_cnf(B, D, (90, 90, 90), dtype=torch.float64, seed=8)
    u0, gout = _inputs(B, D, 3, torch.float64)
    t = torch.tensor([0.0, 0.5, 1.0], dtype=torch.float64)
    argv = ["-ts_rtol", "1e-6", "-ts_atol", "1e-6"]
    a = _mine(argv, func, u0, t, gout, "dopri5", 0.1)
    b = _mine(argv, func, u0, t, gout, "dopri5", 0.1)
    c = _mine(argv + ["-pnode_cnf_save_mb", "0"], func, u0, t, gout, "dopri5", 0.1)
    assert _exact(a[3]) and _exact(b[3]) and _exact(c[3])
    assert a[3]._cb_ex.reused_activations > 0 and c[3]._cb_ex.reused_activations == 0
    _same(a, b)
    _same(a, c)


def test_rk4_training_step_replays_from_a_cuda_graph():
    from pnode import petsc_adjoint

    B, D = 100, 43
    func = cnf_to(exact_cnf(B, D, (86, 86), dtype=torch.float32, seed=2), "cuda")
    Options.clear_all()
    Options.insert_args(FIXED)
    u_static = _inputs(B, D, 2, torch.float32, seed=0)[0].cuda()
    g_static = _inputs(B, D, 2, torch.float32, seed=9)[1].cuda()
    t = torch.tensor([0.0, 1.0], dtype=torch.float64).cuda()
    ode = petsc_adjoint.ODEPetsc()
    ode.setupTS(u_static, func, step_size=0.25, method="rk4", enable_adjoint=True)

    def one_pass():
        return _solve(ode, func, u_static, t, g_static, "cuda")

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            one_pass()
    torch.cuda.current_stream().wait_stream(s)
    assert _exact(ode)
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


def test_past_the_row_limit_takes_the_module_path():
    """(D + 1) B = 65538 rows in fp64 is past one product's reduction length (65535): the exact trace takes the module
    path, while the Hutchinson trace of the same network (2B rows) keeps the evaluator."""
    from pnode import petsc_adjoint

    B, D = 21846, 2
    u0 = _inputs(B, D, 1, torch.float64)[0].cuda()
    kinds = []
    for make in (exact_cnf, CNFFunc):
        func = cnf_to(make(B, D, (16, 16), dtype=torch.float64), "cuda")
        Options.clear_all()
        ode = petsc_adjoint.ODEPetsc()
        ode.setupTS(u0, func, step_size=0.25, method="rk4")
        kinds.append(ode._rhs_kind)
    assert kinds == ["torch", "cnf-net"]
