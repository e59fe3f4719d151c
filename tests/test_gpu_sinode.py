"""SINODE path (BASELINE config 5) on the product's own kernels: the ReLU-MLP right-hand side and its VJP as tensor-core
sliced products (csrc/dense_mlp.cu), the circulant implicit operator and its spectral inverse -- against torch autograd /
dense linear algebra on the same inputs, and the whole ARKIMEX fwd+adjoint pass against the oracle."""
import copy
import os

import pytest
import torch

from oracle import OracleODEPetsc
from pnode_b200.options import Options
from _problems import rel_err
from _workloads import KSExplicit, KSImplicit, ks_dx

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _mlp_pair(n, hidden, dtype, batch, seed=0, out_scale=-1.0, kink_free=False):
    from pnode_b200.densemlp import DenseMlpCallbacks, recognise_relu_mlp

    func = KSExplicit(n, hidden=hidden, dtype=dtype, seed=seed)
    if kink_free:  # every hidden unit active: the fp32 / fp64 comparison at full size involves no ReLU branch decisions
        with torch.no_grad():  # (weights / 5 keep the row sums of W, which multiply the common shift, well below 1)
            for m in list(func.F)[:-1]:
                if isinstance(m, torch.nn.Linear):
                    m.weight.mul_(0.2)
                    m.bias.fill_(1.0)
    func = func.cuda()
    if out_scale > 0:
        func.forward = lambda t, y, F=func.F: F(y)
    meta = torch.empty(batch, n, dtype=dtype, device="cuda")
    spec = recognise_relu_mlp(func, meta)
    assert spec is not None and spec[1] == out_scale
    return func, DenseMlpCallbacks(func, meta.shape, spec[0], spec[1])


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-12), (torch.float32, 1e-4)])  # BASELINE bar: 1e-10 / 1e-4
@pytest.mark.parametrize("n,hidden,batch", [(64, 200, 16), (96, 130, 37), (1024, 3200, 256)])
def test_dense_mlp_forward_and_vjp_match_autograd(dtype, tol, n, hidden, batch):
    # fp32 at full size: 3.3 M hidden units per evaluation, a few of them within fp32 rounding of the ReLU kink; each one that
    # takes the other branch than the fp64 reference moves J^T w by O(1e-3) of its norm (any fp32 implementation does this):
    # that comparison is made with all units active, the ReLU logic at the smaller sizes and in fp64
    func, cb = _mlp_pair(n, hidden, dtype, batch, kink_free=(dtype == torch.float32 and batch >= 256))
    g = torch.Generator().manual_seed(n + batch)
    u = (0.5 * torch.randn(batch, n, generator=g, dtype=torch.float64)).to(dtype).cuda()
    w = torch.randn(batch, n, generator=g, dtype=torch.float64).to(dtype).cuda()
    cb.begin(True, keep=True)
    out = cb.f(0.0, u.reshape(-1), keep=True)
    # reference in fp64 with the same (dtype-rounded) parameters
    f64 = copy.deepcopy(func).double()
    x = u.double().clone().requires_grad_(True)
    ref = f64(0.0, x)
    gr = torch.autograd.grad(ref, [x] + list(f64.parameters()), w.double())
    assert rel_err(out.view(batch, n), ref) < tol
    mu = torch.zeros(cb.nparams, dtype=dtype, device="cuda")
    vu, _ = cb.vjp_accumulate(0.0, u.reshape(-1), w.reshape(-1), mu, 0.37)
    assert cb.reused_activations == 1
    assert rel_err(vu.view(batch, n), gr[0]) < tol
    off = 0
    for p, gp in zip(f64.parameters(), gr[1:]):
        assert rel_err(mu[off:off + p.numel()].view_as(p), 0.37 * gp) < tol, (tuple(p.shape), off)
        off += p.numel()
    # the generic-interface vjp (per-parameter tensors, no kept activation set) gives the same numbers
    cb.release()
    vu2, gps = cb.vjp(0.0, u.reshape(-1).clone(), w.reshape(-1))
    assert rel_err(vu2, vu) < 1e-13 if dtype == torch.float64 else 1e-6
    for gp2, gp in zip(gps, gr[1:]):
        assert rel_err(gp2.view_as(gp), gp) < tol


def test_recognisers_refuse_what_they_cannot_reproduce():
    from pnode_b200.densemlp import recognise_circulant, recognise_relu_mlp

    meta = torch.empty(4, 32, dtype=torch.float64, device="cuda")
    f = KSExplicit(32, hidden=40).cuda()
    assert recognise_relu_mlp(f, meta) is not None
    f.forward = lambda t, y, F=f.F: -F(y) * (1.0 + t)   # time dependent
    assert recognise_relu_mlp(f, meta) is None
    g = KSExplicit(32, hidden=40).cuda()
    g.F[1] = torch.nn.Tanh()                              # not a ReLU chain
    assert recognise_relu_mlp(g, meta) is None
    im = KSImplicit(ks_dx(32)).cuda()
    col = recognise_circulant(im, meta)
    assert col is not None and int((col != 0).sum()) == 5
    im2 = KSImplicit(ks_dx(32)).cuda()
    im2.A.padding_mode = "zeros"                          # Toeplitz, not circulant
    assert recognise_circulant(im2, meta) is None
    im3 = KSImplicit(ks_dx(32)).cuda()
    im3.A.weight.requires_grad_(True)                     # trainable operator: mu_I needs the generic path
    assert recognise_circulant(im3, meta) is None


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-12), (torch.float32, 1e-5)])
@pytest.mark.parametrize("n", [64, 1024])
def test_circulant_operator_and_spectral_inverse(dtype, tol, n):
    from pnode_b200.densemlp import CirculantCallbacks, CirculantSolver, recognise_circulant
    from pnode_b200.device import DeviceOps

    B = 8
    im = KSImplicit(ks_dx(n), dtype=dtype).cuda()
    meta = torch.empty(B, n, dtype=dtype, device="cuda")
    col = recognise_circulant(im, meta)
    cb = CirculantCallbacks(im, meta.shape, col, dtype, meta.device)
    g = torch.Generator().manual_seed(n)
    y = torch.randn(B, n, generator=g, dtype=torch.float64).to(dtype).cuda()
    idx = (torch.arange(n)[:, None] - torch.arange(n)[None, :]) % n
    J = col[idx].cuda()                                    # fp64 dense operator
    assert rel_err(cb.f(0.0, y.reshape(-1)).view(B, n), im(0.0, y)) < tol
    assert rel_err(cb.vjp(0.0, y.reshape(-1), y.reshape(-1))[0].view(B, n), y.double() @ J) < tol
    imp = CirculantSolver(DeviceOps(meta.device, dtype), cb, "torch", B, True)
    imp.reset()
    shift = 1.0 / (0.2 * 0.4358665215)
    A = shift * torch.eye(n, dtype=torch.float64, device="cuda") - J
    Y = imp.solve(0.0, y.reshape(-1), shift, y.reshape(-1)).view(B, n)
    ref = shift * torch.linalg.solve(A, y.double().T).T
    # (shift I - J) has condition number 6e6 at n = 1024 (3e2 at 64): an LU solve is good to cond * eps ~ 1e-9, and so is
    # the spectral inverse; fp32: the operator's entries (1/dx^4) carry 1e-7 themselves
    stol = (1e-11 if n <= 64 else 5e-9) if dtype == torch.float64 else 2e-4
    assert rel_err(Y, ref) < stol
    Yt = imp.solve_transpose(0.0, None, shift, y.reshape(-1)).view(B, n)
    assert rel_err(Yt, torch.linalg.solve(A.T, y.double().T).T) < stol


def _ks_pass(N, H, B, dtype, name="3", seed=4):
    from pnode import petsc_adjoint

    g = torch.Generator().manual_seed(seed)
    u0 = (0.5 * torch.randn(B, N, generator=g, dtype=torch.float64)).to(dtype)
    gout = torch.randn(2, B, N, generator=g, dtype=torch.float64).to(dtype)
    t = torch.tensor([0.0, 0.2], dtype=torch.float64)
    argv = ["-ts_adapt_type", "none", "-snes_type", "ksponly", "-ts_arkimex_type", name]
    Options.clear_all()
    Options.insert_args(argv)
    f_im, f_ex = KSImplicit(ks_dx(N), dtype=dtype).cuda(), KSExplicit(N, hidden=H, dtype=dtype).cuda()
    ode = petsc_adjoint.ODEPetsc()
    ode.setupTS(u0.cuda(), f_im, step_size=0.2, method="imex", imex_form=True, func2=f_ex, batch_size=B,
                linear_solver="torch", fixed_jacobian_across_solves=True)
    y0 = u0.cuda().clone().requires_grad_(True)
    out = ode.odeint_adjoint(y0, t.cuda())
    (out * gout.cuda()).sum().backward()
    mu = torch.cat([p.grad.reshape(-1) for p in f_ex.parameters()])
    return ode, out.detach(), y0.grad, mu, (argv, u0, gout, t)


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-10), (torch.float32, 1e-4)])
@pytest.mark.parametrize("name", ["3", "l2", "ars443", "1bee"])
def test_ks_pass_matches_oracle(dtype, tol, name):
    N, H, B = 64, 200, 16
    ode, out, lam, mu, (argv, u0, gout, t) = _ks_pass(N, H, B, dtype, name)
    assert ode.path == "generic+dense-mlp+circulant-rhs"
    f_im, f_ex = KSImplicit(ks_dx(N), dtype=dtype), KSExplicit(N, hidden=H, dtype=dtype)
    ref = OracleODEPetsc(argv)
    ref.setupTS(u0, f_im, step_size=0.2, method="imex", imex_form=True, func2=f_ex, batch_size=B, linear_solver="torch")
    y0 = u0.clone().requires_grad_(True)
    o = ref.odeint_adjoint(y0, t)
    (o * gout).sum().backward()
    mu_ref = torch.cat([p.grad.reshape(-1) for p in f_ex.parameters()])
    assert rel_err(out, o) < tol and rel_err(lam, y0.grad) < tol and rel_err(mu, mu_ref) < tol, \
        (rel_err(out, o), rel_err(lam, y0.grad), rel_err(mu, mu_ref))


def test_ks_full_size_against_the_committed_oracle_fixture():
    """BASELINE config 5 at full size (N=1024, H=3200, B=256, fp64, ARKIMEX 3, h=0.2): trajectory, lambda and mu against the
    CPU oracle's results for the same seeded inputs (tests/golden/make_cfg5_full.py ran the oracle on the CPU): sampled batch
    rows of the final state and lambda, sampled entries of mu, and sum / norm of all three."""
    path = os.path.join(GOLDEN, "cfg5_full_fp64.pt")
    fx = torch.load(path)
    N, H, B = fx["N"], fx["H"], fx["B"]
    ode, out, lam, mu, _ = _ks_pass(N, H, B, torch.float64, "3", seed=fx["seed"])
    assert ode.path == "generic+dense-mlp+circulant-rhs" and mu.numel() == 37287424
    u, lam, rows = out[-1].cpu(), lam.cpu(), fx["rows"]
    errs = dict(traj=rel_err(u[rows], fx["u_rows"]), lam=rel_err(lam[rows], fx["lam_rows"]),
                mu_sample=rel_err(mu.cpu()[fx["mu_index"]], fx["mu_sample"]))
    for name, key, x in (("traj", "u", u), ("lam", "lam", lam), ("mu", "mu", mu)):
        errs[name + "_sum"] = abs(x.double().sum().item() - fx[key + "_sum"]) / fx[key + "_abs_sum"]
        errs[name + "_norm"] = abs(x.double().norm().item() - fx[key + "_norm"]) / fx[key + "_norm"]
    # (shift I - J) has condition number 6e6 at N = 1024 and the stage right-hand sides are rough (K^I_0 = J u_n ~ 1e7 |u_n|):
    # the reference algorithm itself moves by 1.1e-8 (trajectory) when only the summation order inside f_I changes, by 2.2e-8
    # when the Newton step is replaced by the direct solve (tests/golden/cfg5_noise_floor.py; lambda and mu are piecewise
    # constant in Y and move only through the transposed solves).  Bars: that floor x 5 for the trajectory, 1e-8 for lambda / mu.
    assert errs["traj"] < 1e-7 and errs["lam"] < 1e-8 and errs["mu_sample"] < 1e-8, errs
    assert errs["traj_sum"] < 1e-7 and errs["traj_norm"] < 1e-7, errs
    assert errs["lam_sum"] < 1e-8 and errs["lam_norm"] < 1e-8, errs
    assert errs["mu_sum"] < 1e-8 and errs["mu_norm"] < 1e-8, errs


def test_burgers_pair_takes_the_same_evaluators_and_matches_the_oracle():
    """SURVEY.md 8f.3: the Burgers driver's shapes (Burgers.py:134-195: 3-tap periodic stencil, MLP of width 9N/8 returning
    +net(y), several output times, ARKIMEX 1bee as in run_a100_512.sh) at N = 64, batch 10, against the oracle."""
    from pnode import petsc_adjoint
    from _workloads import BurgersExplicit, BurgersImplicit

    N, B = 64, 10
    g = torch.Generator().manual_seed(8)
    x = torch.linspace(0, 1, N + 1, dtype=torch.float64)[:-1]
    u0 = torch.sin(2 * torch.pi * x)[None, :] * (0.5 + torch.rand(B, 1, generator=g, dtype=torch.float64))
    t = torch.arange(5, dtype=torch.float64) * 0.02
    gout = torch.randn(5, B, N, generator=g, dtype=torch.float64)
    argv = ["-ts_adapt_type", "none", "-snes_type", "ksponly", "-ts_arkimex_type", "1bee"]
    res = []
    for dev in ("cpu", "cuda"):
        Options.clear_all()
        Options.insert_args(argv)
        f_im, f_ex = BurgersImplicit(N).to(dev), BurgersExplicit(N).to(dev)
        ode = OracleODEPetsc(argv) if dev == "cpu" else petsc_adjoint.ODEPetsc()
        ode.setupTS(u0.to(dev), f_im, step_size=0.01, method="imex", imex_form=True, func2=f_ex, batch_size=B,
                    linear_solver="torch")
        y0 = u0.to(dev).clone().requires_grad_(True)
        out = ode.odeint_adjoint(y0, t.to(dev))
        (out * gout.to(dev)).sum().backward()
        res.append((out.detach().cpu(), y0.grad.cpu(), torch.cat([p.grad.reshape(-1) for p in f_ex.parameters()]).cpu(), ode))
    o, p = res
    assert p[3].path == "generic+dense-mlp+circulant-rhs" and p[3]._cb_ex.out_scale == 1.0
    errs = [rel_err(a, b) for a, b in zip(p[:3], o[:3])]
    assert max(errs) < 1e-10, errs
