"""GPU parity of the fused FFJORD CNF sweeps (csrc/cnf_rk.cu through ODEPetsc -> ctypes -> C ABI) against the oracle,
which evaluates the same model the way the reference does (autograd Hutchinson trace, second-order autograd VJP)."""
import copy

import pytest
import torch

from oracle import OracleODEPetsc
from pnode_b200.options import Options
from _problems import rel_err
from _workloads import CNFFunc, cnf_to

pytestmark = pytest.mark.gpu


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
    return out.detach(), y0.grad, [p.grad for p in f.parameters()], ode


def _pair(argv, func, u0, t, gout, method, step, fused=True):
    from pnode import petsc_adjoint

    o = _run(lambda: OracleODEPetsc(argv), "cpu", argv, func, u0, t, gout, method, step)
    p = _run(lambda: petsc_adjoint.ODEPetsc(), "cuda", argv + ([] if fused else ["-pnode_fused", "0"]), func, u0, t, gout,
             method, step)
    return o, p


def _compare(p, o, tol):
    assert rel_err(p[0], o[0]) < tol, ("trajectory", rel_err(p[0], o[0]))
    assert rel_err(p[1], o[1]) < tol, ("lambda", rel_err(p[1], o[1]))
    assert len(p[2]) == len(o[2]) == 10
    for i, (a, b) in enumerate(zip(p[2], o[2])):
        assert rel_err(a, b) < tol, ("mu[%d]" % i, rel_err(a, b))


@pytest.mark.parametrize("dtype,tol,ts_tol", [(torch.float64, 1e-10, "1e-6"), (torch.float32, 1e-4, "1e-4")])
@pytest.mark.parametrize("B", [1000, 77, 20001])  # 20001: past the small-batch kernels (4 lanes per trajectory slot), odd tail
def test_config3_adaptive_dopri5_fused(dtype, tol, ts_tol, B):
    func = CNFFunc(B, 6, (60,), dtype=dtype)
    u0, gout = _inputs(B, 6, 2, dtype)
    t = torch.tensor([0.0, 1.0], dtype=torch.float64)
    o, p = _pair(["-ts_rtol", ts_tol, "-ts_atol", ts_tol], func, u0, t, gout, "dopri5", 0.05)
    assert p[3].path == "fused-cnf-rk"
    lo, lp = o[3].ts.log, p[3]._loop.attempts
    assert [a[2] for a in lo] == [a[2] for a in lp], "accept/reject pattern"
    for a, b in zip(lo, lp):
        assert a[1] == pytest.approx(b[1], rel=1e-8 if dtype == torch.float64 else 2e-2)
    _compare(p, o, tol)


def test_rejections_and_multiple_output_times_fp64():
    B = 200
    func = CNFFunc(B, 6, (60,), dtype=torch.float64, seed=3)
    with torch.no_grad():  # make the dynamics stiffer so that the first big step is rejected
        for prm in func.parameters():
            prm.mul_(4.0)
    u0, gout = _inputs(B, 6, 4, torch.float64)
    t = torch.tensor([0.0, 0.3, 0.35, 1.0], dtype=torch.float64)
    o, p = _pair(["-ts_rtol", "1e-7", "-ts_atol", "1e-7"], func, u0, t, gout, "dopri5", 0.5)
    assert p[3].path == "fused-cnf-rk"
    assert any(not a[2] for a in o[3].ts.log), "case must contain a rejected attempt"
    assert [a[2] for a in o[3].ts.log] == [a[2] for a in p[3]._loop.attempts]
    _compare(p, o, 2e-9)  # weights x4: the flow amplifies rounding differences ~20x more than the default model


@pytest.mark.parametrize("method,argv,t_via_f32", [
    pytest.param("rk4", ["-ts_adapt_type", "none"], True, id="rk4-argv0"),
    pytest.param("dopri5", ["-ts_adapt_type", "none"], True, id="dopri5-argv1"),
    pytest.param("bosh3", [], True, id="bosh3-argv2"),
    pytest.param("euler", [], True, id="euler-argv3"),
    # a module that keeps t in fp64: every stage time but the first is off the fp32 grid
    pytest.param("dopri5", ["-ts_adapt_type", "none"], False, id="dopri5-t-f64")])
def test_other_schemes_fused_fp64(method, argv, t_via_f32):
    B = 64
    func = CNFFunc(B, 6, (60,), dtype=torch.float64, seed=5, t_via_f32=t_via_f32)
    u0, gout = _inputs(B, 6, 3, torch.float64)
    t = torch.tensor([0.0, 0.5, 1.0], dtype=torch.float64) + (0.0 if t_via_f32 else 0.3)
    o, p = _pair(argv, func, u0, t, gout, method, 0.25)
    assert p[3].path == "fused-cnf-rk" and p[3]._fused.spec.t_via_f32 == int(t_via_f32)
    _compare(p, o, 1e-10)


def test_many_steps_grow_the_checkpoint_buffer():
    B = 40
    func = CNFFunc(B, 6, (60,), dtype=torch.float64, seed=9)
    u0, gout = _inputs(B, 6, 2, torch.float64)
    t = torch.tensor([0.0, 1.0], dtype=torch.float64)
    o, p = _pair(["-ts_adapt_type", "none"], func, u0, t, gout, "rk4", 0.02)  # 50 steps > 16 > 32 slots
    assert p[3].path == "fused-cnf-rk" and p[3]._loop.steps == 50
    _compare(p, o, 1e-10)


def test_fused_equals_generic_and_single_time_point():
    B = 500
    func = CNFFunc(B, 6, (60,), dtype=torch.float64, seed=7)
    u0, gout = _inputs(B, 6, 1, torch.float64)
    t = torch.tensor([0.8], dtype=torch.float64)
    argv = ["-ts_rtol", "1e-6", "-ts_atol", "1e-6"]
    o, p = _pair(argv, func, u0, t, gout, "dopri5", 0.1)
    assert p[0].shape == (1, B * 7)
    _compare(p, o, 1e-10)
    _, g = _pair(argv, func, u0, t, gout, "dopri5", 0.1, fused=False)
    assert g[3].path == "generic" and p[3].path == "fused-cnf-rk"
    _compare(p, g, 1e-10)


def test_probe_is_sampled_like_the_reference_when_absent():
    """odefunc.py:359-364: `_e` is drawn inside the first RHS evaluation of a solve; the fused path draws it instead."""
    from pnode import petsc_adjoint

    B = 32
    func = cnf_to(CNFFunc(B, 6, (60,), dtype=torch.float32), "cuda")
    func.base_func.before_odeint()  # e <- None
    Options.insert_args(["-ts_adapt_type", "none"])
    u0, _ = _inputs(B, 6, 2, torch.float32)
    ode = petsc_adjoint.ODEPetsc()
    ode.setupTS(u0.cuda(), func, step_size=0.25, method="rk4")
    out = ode.odeint_adjoint(u0.cuda(), torch.tensor([0.0, 1.0]).cuda())
    assert ode.path == "fused-cnf-rk" and func.base_func._e is not None and func.base_func._e.shape == (B, 6)
    # the same probe through the un-fused module gives the same answer
    Options.insert_args(["-pnode_fused", "0"])
    ode2 = petsc_adjoint.ODEPetsc()
    ode2.setupTS(u0.cuda(), func, step_size=0.25, method="rk4")
    out2 = ode2.odeint_adjoint(u0.cuda(), torch.tensor([0.0, 1.0]).cuda())
    assert ode2.path == "generic" and rel_err(out, out2) < 1e-5


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_device_controller_follows_the_host_controller(dtype):
    """The accept/reject verdict and the next step size taken by the attempt kernel's last block (csrc/cnf_rk.cu, namespace
    ctl) against the host TimeLoop fed the same kernel's error norm once per attempt: same attempts, same steps, same
    output-time copies.  The case has rejected attempts, clamped steps and three output times.  The attempts run in the
    CUDA-graph WHILE loop (one launch per solve)."""
    from pnode import petsc_adjoint

    B = 300
    func = CNFFunc(B, 6, (60,), dtype=dtype, seed=3)
    with torch.no_grad():
        for prm in func.parameters():
            prm.mul_(4.0)
    u0, gout = _inputs(B, 6, 4, dtype)
    t = torch.tensor([0.0, 0.3, 0.35, 1.0], dtype=torch.float64)
    tol = "1e-7" if dtype == torch.float64 else "1e-4"
    argv = ["-ts_rtol", tol, "-ts_atol", tol]
    d = _run(lambda: petsc_adjoint.ODEPetsc(), "cuda", argv, func, u0, t, gout, "dopri5", 0.5)
    h = _run(lambda: petsc_adjoint.ODEPetsc(), "cuda", argv + ["-pnode_device_controller", "0"], func, u0, t, gout, "dopri5",
             0.5)
    assert d[3].path == h[3].path == "fused-cnf-rk"
    assert d[3]._fused.device_controller and not h[3]._fused.device_controller
    la, lb = d[3]._loop.attempts, h[3]._loop.attempts
    if dtype == torch.float64:
        assert any(not a[2] for a in la), "case must contain a rejected attempt"
    assert [a[2] for a in la] == [a[2] for a in lb]
    # same kernel, same inputs; the step factor differs by the rounding of pow() on the two sides, and one ulp of h moves the
    # NEXT error norm (a difference of nearly equal fp numbers) by ~eps/tol relative
    rel = 1e-8 if dtype == torch.float64 else 2e-2
    for a, b in zip(la, lb):
        assert a[0] == pytest.approx(b[0], rel=rel, abs=1e-15) and a[1] == pytest.approx(b[1], rel=rel)
    assert d[3]._loop.cur_sol_steps == h[3]._loop.cur_sol_steps
    _compare(d, h, 1e-11 if dtype == torch.float64 else 1e-4)


def test_device_controller_many_steps_and_single_end_time():
    """More accepted steps than the checkpoint buffer starts with (the device loop stops with done = 4, the host doubles
    the buffer and the loop goes on); one-element t (no span); two solves in a row on the same object (buffers and the
    cached loop graph are reused).  Compared with the host-controlled run of the same kernels (at this tolerance the
    error estimate is too close to rounding noise for the oracle's autograd evaluation to take the same decisions)."""
    from pnode import petsc_adjoint
    from pnode_b200.fused import FusedCnfRK

    B = 64
    func = CNFFunc(B, 6, (60,), dtype=torch.float64, seed=11)
    u0, gout = _inputs(B, 6, 1, torch.float64)
    t = torch.tensor([1.0], dtype=torch.float64)
    argv = ["-ts_rtol", "1e-10", "-ts_atol", "1e-10"]
    room = FusedCnfRK.CKPT_STEPS0
    FusedCnfRK.CKPT_STEPS0 = 2
    try:
        d = _run(lambda: petsc_adjoint.ODEPetsc(), "cuda", argv, func, u0, t, gout, "dopri5", 0.01)
        ode = d[3]
        y0 = u0.to("cuda").clone().requires_grad_(True)
        again = ode.odeint_adjoint(y0, t.to("cuda"))  # same object: pooled checkpoint buffer, cached graph
        lam_again, = torch.autograd.grad((again * gout.to("cuda")).sum(), [y0])
    finally:
        FusedCnfRK.CKPT_STEPS0 = room
    h = _run(lambda: petsc_adjoint.ODEPetsc(), "cuda", argv + ["-pnode_device_controller", "0"], func, u0, t, gout, "dopri5",
             0.01)
    assert d[3].path == "fused-cnf-rk" and d[3]._fused.device_controller and not h[3]._fused.device_controller
    assert d[3]._loop.steps > 4
    assert d[3]._loop.steps == h[3]._loop.steps
    assert d[0].shape == (1, B * 7)
    _compare(d, h, 1e-9)
    assert torch.equal(again.detach(), d[0]) and torch.equal(lam_again, d[1])


def test_device_controller_reports_divergence():
    """[PETSc] TS_DIVERGED_STEP_REJECTED after more than -ts_adapt max_reject consecutive rejections."""
    from pnode import petsc_adjoint

    B = 32
    func = CNFFunc(B, 6, (60,), dtype=torch.float64, seed=3)
    with torch.no_grad():
        for prm in func.parameters():
            prm.mul_(40.0)
    u0, gout = _inputs(B, 6, 2, torch.float64)
    t = torch.tensor([0.0, 1.0], dtype=torch.float64)
    argv = ["-ts_rtol", "1e-13", "-ts_atol", "1e-13", "-ts_max_reject", "2"]
    with pytest.raises(RuntimeError, match="TS_DIVERGED_STEP_REJECTED"):
        _run(lambda: petsc_adjoint.ODEPetsc(), "cuda", argv, func, u0, t, gout, "dopri5", 1.0)


@pytest.mark.parametrize("extra", [[], ["-pnode_device_controller", "0"]], ids=["device-loop", "host-loop"])
def test_backward_sees_the_probe_of_its_own_forward(extra):
    """FFJORD draws a fresh Hutchinson probe per forward (cnf.py: odefunc.before_odeint).  Two forwards with different
    probes, then the two backwards in reverse order, on ONE ODEPetsc object: each must equal the solve done on its own
    (the probe and the checkpoints of a solve travel with its autograd state, csrc buffers are pooled, not shared)."""
    from pnode import petsc_adjoint

    B = 48
    func = cnf_to(CNFFunc(B, 6, (60,), dtype=torch.float64, seed=5), "cuda")
    probes = [torch.randn(B, 6, generator=torch.Generator().manual_seed(s), dtype=torch.float64).cuda() for s in (1, 2)]
    u0s = [_inputs(B, 6, 2, torch.float64, seed=s)[0].cuda() for s in (3, 4)]
    gout = _inputs(B, 6, 2, torch.float64)[1].cuda()
    t = torch.tensor([0.0, 1.0], dtype=torch.float64).cuda()
    Options.clear_all()
    Options.insert_args(["-ts_rtol", "1e-7", "-ts_atol", "1e-7"] + extra)

    def solve(ode, k):
        func.base_func.before_odeint(e=probes[k])
        y0 = u0s[k].clone().requires_grad_(True)
        return y0, ode.odeint_adjoint(y0, t)

    alone = []
    for k in (0, 1):
        ode = petsc_adjoint.ODEPetsc()
        ode.setupTS(u0s[k], func, step_size=0.05, method="dopri5", enable_adjoint=True)
        func.zero_grad(set_to_none=True)
        y0, out = solve(ode, k)
        (out * gout).sum().backward()
        alone.append((out.detach().clone(), y0.grad.clone(), [p.grad.clone() for p in func.parameters()]))
    ode = petsc_adjoint.ODEPetsc()
    ode.setupTS(u0s[0], func, step_size=0.05, method="dopri5", enable_adjoint=True)
    ya, outa = solve(ode, 0)
    yb, outb = solve(ode, 1)
    assert ode.path == "fused-cnf-rk" and ode._fused.device_controller == (not extra)
    for k, (y0, out) in ((1, (yb, outb)), (0, (ya, outa))):  # backwards in reverse order
        func.zero_grad(set_to_none=True)
        (out * gout).sum().backward()
        assert torch.equal(out.detach(), alone[k][0]) and torch.equal(y0.grad, alone[k][1])
        for a, b in zip([p.grad for p in func.parameters()], alone[k][2]):
            assert torch.equal(a, b)


@pytest.mark.parametrize("seed", range(24))
def test_device_step_controller_takes_the_host_controller_s_decisions(seed):
    """csrc/cnf_rk.cu namespace ctl against controller.TimeLoop on random error-norm sequences (pnode_cnf_ctl_probe runs the
    code the attempt kernel's last block runs): verdicts, times, next step sizes (MATCHSTEP clamp / halving / restore after
    an output-time hit), span counters and output slots -- branches a handful of real solves does not reach."""
    import ctypes as C
    import random

    from pnode_b200 import _lib
    from pnode_b200.controller import TimeLoop

    rng = random.Random(seed)
    lib = _lib.load()
    nspan = rng.choice([0, 2, 3, 5, 9])
    if nspan:
        times = sorted(rng.uniform(0.0, 2.0) for _ in range(nspan))
        if rng.random() < 0.5:
            times[1] = times[0] + 1e-3  # a very short first interval
    else:
        times = [rng.uniform(0.3, 2.0)]
    h0 = rng.choice([1e-3, 0.05, 0.4, 5.0])
    order = rng.choice([3, 5])
    double = rng.random() < 0.5
    loop = TimeLoop(times, h0, True, order, double, max_reject=10)
    n_global = 1000.0
    c = _lib.CnfCtl()
    c.t, c.h, c.t_end = loop.t, loop.h, loop.t_end
    for i in range(nspan):
        c.span[i] = loop.span[i]
    c.n_global, c.delta = n_global, loop.delta
    c.nspan, c.order, c.max_reject = nspan, order, 10
    c.done = 1 if loop.done else 0
    c.prev_ok, c.ctr, c.cur_sol_index, c.pending_slot = 1, 1, 1, -1
    enorms = []
    slots = []
    for _ in range(600):  # the host controller on a random walk of error norms, mostly accepted
        if loop.done:
            break
        e = rng.choice([0.0, 1e-6, 0.05, 0.3, 0.8, 0.999, 1.0, 1.0001, 1.5, 4.0, 50.0]) if rng.random() < 0.3 else \
            rng.lognormvariate(-0.7, 0.8)
        enorms.append(e)
        try:
            if loop.report(e):
                slots.append(loop.last_out_slot)
        except RuntimeError:
            break
    sumsq = torch.tensor([e * e * n_global for e in enorms], dtype=torch.float64, device="cuda")
    dev = torch.frombuffer(bytearray(bytes(c)), dtype=torch.uint8).cuda()
    _lib.check(lib.pnode_cnf_ctl_probe(dev.data_ptr(), sumsq.data_ptr(), len(enorms), None))
    torch.cuda.synchronize()
    got = _lib.CnfCtl.from_buffer_copy(dev.cpu().numpy().tobytes())
    assert got.attempts == len(loop.attempts)
    for a in range(got.attempts):
        t, h, ok, _ = loop.attempts[a]
        assert bool(got.log_accepted[a]) == ok, a
        assert got.log_t[a] == pytest.approx(t, rel=1e-13, abs=1e-15) and got.log_h[a] == pytest.approx(h, rel=1e-12), a
    assert got.steps == loop.steps and got.ctr == loop.ctr and got.cur_sol_index == loop.cur_sol_index
    assert got.t == pytest.approx(loop.t, rel=1e-13, abs=1e-15)
    if loop.done:
        assert got.done == 1
    elif loop._rejections > loop.max_reject:
        assert got.done == 2
    else:
        assert got.done == 0 and got.h == pytest.approx(loop.h, rel=1e-12)
