"""csrc/conv_block.cu through the C ABI (pnode_convblock_forward / pnode_convblock_vjp) against the stock torch module and its
autograd backward on the same inputs: the whole SqueezeNext ODE-block right-hand side (convolutions + train-mode BatchNorm + ReLU),
its state VJP, every parameter gradient, and the BatchNorm side effects.  fp64: 1e-10; fp32: 1e-4 (IEEE fp32 library reference)."""
import copy
import ctypes as C

import pytest
import torch

from _problems import rel_err
from _workloads import OdeConvBlock

pytestmark = pytest.mark.gpu


def _callbacks(func, shape):
    from pnode_b200.convblock import ConvBlockCallbacks
    from pnode_b200.options import Options

    Options.insert_args(["-pnode_convblock_native", "1"])  # also below the pixel count where "auto" prefers library GEMMs
    cb = ConvBlockCallbacks(func, torch.Size(shape))
    assert cb.native, "the conv-block kernels must accept this shape"
    return cb


def _reference(func, x, w):
    f = copy.deepcopy(func)
    xr = x.clone().requires_grad_(True)
    out = f(0.0, xr)
    out.backward(w)
    return out.detach(), xr.grad, [p.grad for p in f.parameters()], f


# (N, C, H, W): full tiles, partial tiles / partial warps, one-lane rows, the four CIFAR block aspect ratios (scaled down)
SHAPES = [(16, 32, 8, 8), (3, 16, 6, 8), (2, 16, 4, 4), (5, 32, 16, 32), (4, 64, 16, 16), (8, 128, 8, 8), (16, 256, 4, 4),
          (1, 16, 1, 4), (2, 32, 3, 64)]


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-10), (torch.float32, 1e-4)])
def test_rhs_and_vjp_match_torch(shape, dtype, tol):
    N, Cc, H, W = shape
    tf32 = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        func = OdeConvBlock(Cc, dtype=dtype, seed=N).cuda()
        with torch.no_grad():  # non-trivial affine parameters and biases
            g = torch.Generator().manual_seed(7)
            for m in func.modules():
                if isinstance(m, torch.nn.BatchNorm2d):
                    m.weight.copy_((torch.rand(m.num_features, generator=g, dtype=torch.float64) + 0.5).to(dtype))
                    m.bias.copy_((0.3 * torch.randn(m.num_features, generator=g, dtype=torch.float64)).to(dtype))
        g = torch.Generator().manual_seed(11)
        x = torch.randn(shape, generator=g, dtype=torch.float64).to(dtype).cuda()
        w = torch.randn(shape, generator=g, dtype=torch.float64).to(dtype).cuda()
        out_r, vu_r, gp_r, f_r = _reference(func, x, w)
        mine = copy.deepcopy(func)
        cb = _callbacks(mine, shape)
        out = cb.f(0.0, x.reshape(-1)).view(shape)
        vu, gp = cb.vjp(0.0, x.reshape(-1), w.reshape(-1))  # reuses the activation set the forward evaluation kept
        assert cb.reused_activations == 1
        cb.begin(True)  # forget it: the same VJP now re-evaluates the forward inside the call, bit-identically
        vu2, gp2 = cb.vjp(0.0, x.reshape(-1), w.reshape(-1))
        assert cb.reused_activations == 1
        assert torch.equal(vu, vu2) and all(torch.equal(a, b) for a, b in zip(gp, gp2))
        torch.cuda.synchronize()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    assert rel_err(out, out_r) < tol, ("f", rel_err(out, out_r))
    assert rel_err(vu.view(shape), vu_r) < tol * 10, ("J^T w", rel_err(vu.view(shape), vu_r))
    flat = lambda gs: torch.cat([q.detach().double().reshape(-1) for q in gs])
    assert rel_err(flat(gp), flat(gp_r)) < tol * 10, ("Jp^T w", rel_err(flat(gp), flat(gp_r)))
    names = [n for n, _ in mine.named_parameters()]
    for n, a, b in zip(names, gp, gp_r):
        if n.endswith("conv1.bias") or ".bias" in n and "conv" in n:
            continue  # a conv bias feeding a BatchNorm has an exactly-zero gradient: rounding noise on both sides
        assert rel_err(a.view_as(b), b) < tol * 50, (n, rel_err(a.view_as(b), b))
    # side effects: f advanced the statistics once, each vjp (forward re-evaluation, replayed or real) once more
    assert int(mine.bn3.num_batches_tracked) == 3 and int(f_r.bn3.num_batches_tracked) == 1
    again = copy.deepcopy(func)
    again(0.0, x), again(0.0, x), again(0.0, x)
    for k in range(1, 6):
        a, b = getattr(mine, "bn%d" % k), getattr(again, "bn%d" % k)
        assert rel_err(a.running_mean, b.running_mean) < tol * 10 and rel_err(a.running_var, b.running_var) < tol * 10


def test_fused_stage_combination_and_mu_accumulation():
    """pnode_convblock_forward with d_base (Y = base_coef*base + k_coef*f(x), k = f(x)) and pnode_convblock_vjp accumulating
    coef * Jp^T w into an existing mu: the two fusions the RK stage loop uses."""
    shape = (4, 32, 8, 16)
    dtype = torch.float64
    func = OdeConvBlock(shape[1], dtype=dtype).cuda()
    g = torch.Generator().manual_seed(5)
    x = torch.randn(shape, generator=g, dtype=dtype).cuda()
    base = torch.randn(shape, generator=g, dtype=dtype).cuda()
    w = torch.randn(shape, generator=g, dtype=dtype).cuda()
    out_r, vu_r, gp_r, _ = _reference(func, x, w)
    cb = _callbacks(copy.deepcopy(func), shape)
    y, k = torch.empty_like(x), torch.empty_like(x)
    cb._native_f(x.reshape(-1), out=y, base=base, base_coef=1.0, k_coef=0.5, k=k)
    assert rel_err(k, out_r) < 1e-10 and rel_err(y, base + 0.5 * out_r) < 1e-10
    mu0 = torch.randn(cb.nparams, generator=g, dtype=dtype).cuda()
    mu = mu0.clone()
    vu, none = cb.vjp_accumulate(0.0, x.reshape(-1), w.reshape(-1), mu, 0.25)
    assert none is None and rel_err(vu.view(shape), vu_r) < 1e-9
    want = mu0 + 0.25 * torch.cat([q.reshape(-1) for q in gp_r])
    assert rel_err(mu, want) < 1e-9
    # bit-reproducible: the same call twice gives identical bits (fixed-order reductions everywhere)
    mu2 = mu0.clone()
    vu2, _ = cb.vjp_accumulate(0.0, x.reshape(-1), w.reshape(-1), mu2, 0.25)
    assert torch.equal(vu, vu2) and torch.equal(mu, mu2)


def test_full_size_properties_of_config4():
    """BASELINE config 4 at its full size ([256,32,32,32], where the CPU oracle takes minutes): size-independent properties.
    (1) batch-permutation equivariance: BatchNorm statistics are sums over the batch, everything else is per sample;
    (2) the VJP is linear in the cotangent and `mu += coef * Jp^T w` accumulates;
    (3) adjoint dot-product test in fp64: <w, (f(x + e v) - f(x - e v)) / 2e> == <J^T w, v> (central differences of the forward
        kernels against the hand-written backward kernels);
    (4) the stock torch module and its autograd backward at the full size, fp64, every parameter gradient."""
    shape = (256, 32, 32, 32)
    g = torch.Generator().manual_seed(21)
    func = OdeConvBlock(32, dtype=torch.float32).cuda()
    cb = _callbacks(func, shape)
    x = torch.randn(shape, generator=g).cuda().reshape(-1)
    w1 = torch.randn(shape, generator=g).cuda().reshape(-1)
    w2 = torch.randn(shape, generator=g).cuda().reshape(-1)
    perm = torch.randperm(shape[0], generator=g).cuda()
    fx = cb.f(0.0, x).view(shape)
    fp = cb.f(0.0, x.view(shape)[perm].contiguous().reshape(-1)).view(shape)
    assert rel_err(fp, fx[perm]) < 2e-6
    va, ga = cb.vjp(0.0, x, w1)
    vb, gb = cb.vjp(0.0, x, w2)
    vc, gc = cb.vjp(0.0, x, (2.0 * w1 - 0.5 * w2))
    flat = lambda gs: torch.cat([q.reshape(-1) for q in gs])
    assert rel_err(vc, 2.0 * va - 0.5 * vb) < 1e-5 and rel_err(flat(gc), 2.0 * flat(ga) - 0.5 * flat(gb)) < 1e-4
    mu = torch.ones(cb.nparams, device="cuda")
    cb.vjp_accumulate(0.0, x, w1, mu, 0.5)
    assert rel_err(mu, 1.0 + 0.5 * flat(ga)) < 1e-6
    # (3) fp64
    func64 = OdeConvBlock(32, dtype=torch.float64).cuda()
    cb64 = _callbacks(func64, shape)
    x64, w64 = x.double(), w1.double()
    v64 = torch.randn(shape, generator=g, dtype=torch.float64).cuda().reshape(-1)
    eps = 1e-8  # millions of ReLU kinks: central differences only settle below ~1e-7 (tools/diag_fd.py, same for the torch module)
    jtw, gp = cb64.vjp(0.0, x64, w64)
    fd = (cb64.f(0.0, x64 + eps * v64) - cb64.f(0.0, x64 - eps * v64)) / (2 * eps)
    lhs, rhs = float(torch.dot(w64, fd)), float(torch.dot(jtw, v64))
    assert abs(lhs - rhs) <= 1e-4 * max(abs(lhs), abs(rhs)), (lhs, rhs)
    # (4) and, since the stock module runs at this size on the GPU in seconds, the direct comparison in fp64
    tf32 = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        out_r, vu_r, gp_r, _ = _reference(func64, x64.view(shape), w64.view(shape))
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    assert rel_err(cb64.f(0.0, x64).view(shape), out_r) < 1e-12 and rel_err(jtw.view(shape), vu_r) < 1e-12
    for (n, _), a, b in zip(func64.named_parameters(), gp, gp_r):
        if not (n.startswith("conv") and n.endswith("bias")):
            assert rel_err(a.view_as(b), b) < 1e-11, (n, rel_err(a.view_as(b), b))


def test_unsupported_shapes_are_refused_by_the_abi_not_computed_wrongly():
    from pnode_b200 import _lib

    lib = _lib.load()
    d = _lib.ConvBlockDesc()
    d.nlayers, d.dtype, d.N, d.H, d.W = 1, 0, 2, 8, 12  # W not a power of two
    l = d.layer[0]
    l.cin = l.cout = 8
    l.kh = l.kw = 1
    l.d_weight = l.d_bias = l.d_gamma = l.d_beta = 16
    assert lib.pnode_convblock_work_bytes(C.byref(d)) == -1
    assert b"power of two" in lib.pnode_last_error()
    d.W = 8
    l.kh = l.kw = 3
    l.ph = l.pw = 1
    assert lib.pnode_convblock_work_bytes(C.byref(d)) == -1


def test_exact_accumulator_is_exact_and_order_independent():
    """The 128-bit fixed-point accumulator behind the BatchNorm statistics: a million adds in whatever order the hardware
    schedules them give the exact sum (math.fsum) to a few ulp of the final conversion, bit-identically on every repetition -- also when the terms
    cancel catastrophically; non-finite terms poison the result instead of disappearing."""
    import math

    from pnode_b200 import _lib

    lib = _lib.load()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    work = torch.zeros(256, dtype=torch.uint8, device="cuda")
    out = torch.zeros(1, dtype=torch.float64, device="cuda")
    g = torch.Generator().manual_seed(0)
    n = 1 << 20
    cases = [torch.randn(n, generator=g, dtype=torch.float64) * 1e3,
             torch.cat((torch.full((n // 2,), 1e15, dtype=torch.float64), torch.full((n // 2,), -1e15, dtype=torch.float64),
                        torch.tensor([2.0 ** -40, -3.5, 7.25], dtype=torch.float64))),
             torch.rand(n, generator=g, dtype=torch.float64) * 2.0 ** -30 - 2.0 ** -31]
    for v in cases:
        want = math.fsum(math.trunc(x * 2.0 ** 60) * 2.0 ** -60 for x in v.tolist()) if float(v.abs().max()) < 1.0 else None
        vd = v.cuda()
        got = []
        for _ in range(3):
            _lib.check(lib.pnode_acc128_probe(vd.data_ptr(), vd.numel(), out.data_ptr(), work.data_ptr(), st))
            got.append(float(out.item()))
        assert got[0] == got[1] == got[2]
        exact = math.fsum(v.tolist())
        if want is not None:  # terms finer than the 2^-60 resolution are truncated toward zero, deterministically; the read-back
            assert abs(got[0] - want) <= 8 * math.ulp(want), (got[0], want)  # rounds each of the 4 replicas to double once
        else:
            assert abs(got[0] - exact) <= v.numel() * 2.0 ** -60 + 4 * math.ulp(exact), (got[0], exact)
    bad = torch.tensor([1.0, float("inf"), 2.0], dtype=torch.float64).cuda()
    _lib.check(lib.pnode_acc128_probe(bad.data_ptr(), 3, out.data_ptr(), work.data_ptr(), st))
    assert math.isnan(float(out.item()))


@pytest.mark.parametrize("name,dtype,tol", [("fp64", torch.float64, 1e-10), ("fp32", torch.float32, 1e-4),
                                            ("fp32_kinkfree", torch.float32, 1e-4)])
def test_config4_full_size_against_the_committed_oracle_fixture(name, dtype, tol):
    """BASELINE config 4 at FULL size ([256,32,32,32], RK4, t=[1.0], one step of h=1) through the drop-in against the CPU
    oracle's results for the same seeded inputs (tests/golden/make_cfg4_full.py): sampled entries + norms of the final state
    and of lambda, mu in full, BatchNorm running statistics, evaluation count."""
    import os

    from pnode import petsc_adjoint
    from pnode_b200.options import Options

    fx = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cfg4_full_%s.pt" % name))
    B, Cc, HW = fx["B"], fx["C"], fx["HW"]
    g = torch.Generator().manual_seed(fx["seed"])
    u0 = torch.randn(B, Cc, HW, HW, generator=g, dtype=torch.float64).to(dtype).cuda()
    gout = torch.randn(1, B, Cc, HW, HW, generator=g, dtype=torch.float64).to(dtype).cuda()
    t = torch.tensor([1.0], dtype=torch.float64).cuda()
    Options.clear_all()
    Options.insert_args(["-ts_adapt_type", "none"])
    func = OdeConvBlock(Cc, dtype=dtype)
    if name.endswith("kinkfree"):
        with torch.no_grad():
            for m in func.modules():
                if isinstance(m, torch.nn.BatchNorm2d):
                    m.bias.copy_(8.0 * m.weight)
    func = func.cuda()
    ode = petsc_adjoint.ODEPetsc()
    ode.setupTS(u0, func, step_size=1.0, method="rk4")
    y0 = u0.clone().requires_grad_(True)
    out = ode.odeint_adjoint(y0, t)
    (out * gout).sum().backward()
    assert ode.path == "generic+convblock-rhs" and ode._cb_im.native
    uf, lam = out[-1].detach().reshape(-1).cpu(), y0.grad.reshape(-1).cpu()
    mu = torch.cat([p.grad.reshape(-1) for p in func.parameters()]).cpu()
    idx = fx["index"]
    errs = dict(u=float((uf[idx] - fx["u_sample"]).abs().max() / fx["u_absmax"]),
                lam=float((lam[idx] - fx["lam_sample"]).abs().max() / fx["lam_absmax"]),
                u_norm=abs(float(uf.double().norm()) - fx["u_norm"]) / fx["u_norm"],
                lam_norm=abs(float(lam.double().norm()) - fx["lam_norm"]) / fx["lam_norm"],
                mu=rel_err(mu, fx["mu"]),
                bn1_mean=rel_err(func.bn1.running_mean.cpu(), fx["bn1_running_mean"]),
                bn5_var=rel_err(func.bn5.running_var.cpu(), fx["bn5_running_var"]))
    assert func.nfe == fx["nfe"]
    if name == "fp32":
        # stock initialisation in fp32: ~23 M ReLU inputs per evaluation, a handful within fp32 rounding of the kink; the state
        # (ReLU is continuous) and the BatchNorm buffers hold the bar, lambda / mu carry those units' O(1e-3) branch effect
        # (the kink-free fixture checks the same arithmetic at 1e-4)
        assert max(errs[k] for k in ("u", "u_norm", "bn1_mean", "bn5_var")) < tol, errs
        assert max(errs[k] for k in ("lam", "lam_norm", "mu")) < 2e-2, errs
    else:
        assert max(errs.values()) < tol, errs

