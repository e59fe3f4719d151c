"""The three non-spiral workloads of BASELINE.json, re-implemented from their definitions in the reference (same math,
same parameter shapes and initialisation) so that parity tests and bench_configs.py can build them without importing
/root/reference:
  * CNFFunc      -- FFJORD tabular CNF right-hand side: ODEnet of ConcatSquashLinear + softplus, Hutchinson trace with a
                    fixed noise sample, state flattened as cat(z.view(-1), logp.view(-1))
                    (ffjord-pnode/lib/layers/diffeq_layers/basic.py:76-86, odefunc.py:53-57,322-385, cnf.py:72-93,140-150)
  * OdeConvBlock -- the SqueezeNext ODE block of examples-pnode/models/sqnxt_PETSc.py:70-121 (five conv+BN+ReLU layers)
  * KSImplicit / KSExplicit -- the SINODE IMEX pair of examples-sinode/KS/models/imex.py:6-70 (fixed circular 5-tap
                    stencil, 5-layer ReLU MLP returning -F(y))
"""
import math

import torch
import torch.nn as nn
import torch.nn.functional as F


class ConcatSquashLinear(nn.Module):
    def __init__(self, dim_in, dim_out):
        super().__init__()
        self._layer = nn.Linear(dim_in, dim_out)
        self._hyper_bias = nn.Linear(1, dim_out, bias=False)
        self._hyper_gate = nn.Linear(1, dim_out)

    def forward(self, t, x):
        return self._layer(x) * torch.sigmoid(self._hyper_gate(t.view(1, 1))) + self._hyper_bias(t.view(1, 1))


class ODEnet(nn.Module):
    """lib/layers/odefunc.py:97-204 restricted to linear ConcatSquash layers + softplus (train_tabular.py defaults);
    same attribute names as the reference (`layers`, `activation_fns`)."""

    def __init__(self, hidden_dims, dim):
        super().__init__()
        dims = [dim] + list(hidden_dims) + [dim]
        self.layers = nn.ModuleList([ConcatSquashLinear(a, b) for a, b in zip(dims[:-1], dims[1:])])
        self.activation_fns = nn.ModuleList([nn.Softplus() for _ in hidden_dims])

    def forward(self, t, y):
        dx = y
        for i, layer in enumerate(self.layers):
            dx = layer(t, dx)
            if i < len(self.layers) - 1:
                dx = self.activation_fns[i](dx)
        return dx


def divergence_approx(f, y, e=None):
    e_dzdx = torch.autograd.grad(f, y, e, create_graph=True)[0]
    return (e_dzdx * e).view(y.shape[0], -1).sum(dim=1)


class ODEfunc(nn.Module):
    """lib/layers/odefunc.py:322-385: dy = diffeq(t, y), dlogp = -Hutchinson trace with noise fixed per solve."""

    def __init__(self, diffeq):
        super().__init__()
        self.diffeq = diffeq
        self.residual = False
        self.rademacher = False
        self.divergence_fn = divergence_approx
        self.register_buffer("_num_evals", torch.tensor(0.0))
        self._e = None

    def before_odeint(self, e=None):
        self._e = e
        self._num_evals.fill_(0)

    def forward(self, t, states):
        y = states[0]
        self._num_evals += 1
        t = torch.tensor(t).type_as(y)
        if self._e is None:
            self._e = torch.randn_like(y)
        with torch.set_grad_enabled(True):
            y.requires_grad_(True)
            dy = self.diffeq(t, y)
            divergence = self.divergence_fn(dy, y, e=self._e).view(y.shape[0], 1)
        return (dy, -divergence)


class ODEfuncT64(ODEfunc):
    """ODEfunc that keeps t in double precision (the reference's module rounds it through float32)."""

    def forward(self, t, states):
        y = states[0]
        self._num_evals += 1
        t = torch.tensor(t, dtype=torch.float64).type_as(y)
        if self._e is None:
            self._e = torch.randn_like(y)
        with torch.set_grad_enabled(True):
            y.requires_grad_(True)
            dy = self.diffeq(t, y)
            divergence = self.divergence_fn(dy, y, e=self._e).view(y.shape[0], 1)
        return (dy, -divergence)


class FlattenFunc(nn.Module):
    """lib/layers/cnf.py:123-150: the state handed to ODEPetsc is cat(z.view(-1), logp.view(-1))."""

    def __init__(self, base_func, y0):
        super().__init__()
        self.base_func = base_func
        self.y0 = y0

    def forward(self, t, y):
        parts, idx = [], 0
        for x0 in self.y0:
            parts.append(y[idx: idx + x0.numel()].view(*x0.shape))
            idx += x0.numel()
        out = self.base_func(t, tuple(parts))
        return torch.cat([o.contiguous().view(-1) for o in out])


def CNFFunc(batch, dim=6, hidden_dims=(60,), dtype=torch.float32, seed=0, device="cpu", t_via_f32=True):
    """FlattenFunc(ODEfunc(ODEnet)) with the Hutchinson probe already fixed (seeded) -- what cnf.py:72-80 builds.  With
    t_via_f32=False the ODEfunc keeps t in double precision (ODEfuncT64) instead of rounding it through float32."""
    torch.manual_seed(seed)
    odefunc = (ODEfunc if t_via_f32 else ODEfuncT64)(ODEnet(hidden_dims, dim).to(dtype))
    g = torch.Generator().manual_seed(seed + 1)
    odefunc._e = torch.randn(batch, dim, generator=g, dtype=torch.float64).to(dtype)
    y0 = (torch.zeros(batch, dim, dtype=dtype), torch.zeros(batch, 1, dtype=dtype))
    return FlattenFunc(odefunc, y0)


def cnf_to(func, device):
    """Move a CNFFunc (module + the probe/y0 tensors that are plain attributes, as in the reference) to a device."""
    func = func.to(device)
    func.base_func._e = func.base_func._e.to(device)
    func.y0 = tuple(x.to(device) for x in func.y0)
    return func


class OdeConvBlock(nn.Module):
    def __init__(self, dim, dtype=torch.float32, seed=0):
        super().__init__()
        torch.manual_seed(seed)
        r = dim // 2
        self.conv1 = nn.Conv2d(dim, r, 1, 1, bias=True)
        self.bn1 = nn.BatchNorm2d(r)
        self.conv2 = nn.Conv2d(r, r // 2, 1, 1, bias=True)
        self.bn2 = nn.BatchNorm2d(r // 2)
        self.conv3 = nn.Conv2d(r // 2, r, (1, 3), 1, (0, 1), bias=True)
        self.bn3 = nn.BatchNorm2d(r)
        self.conv4 = nn.Conv2d(r, r, (3, 1), 1, (1, 0), bias=True)
        self.bn4 = nn.BatchNorm2d(r)
        self.conv5 = nn.Conv2d(r, dim, 1, 1, bias=True)
        self.bn5 = nn.BatchNorm2d(dim)
        self.to(dtype)
        self.nfe = 0

    def forward(self, t, x):
        self.nfe += 1
        out = F.relu(self.bn1(self.conv1(x)))
        out = F.relu(self.bn2(self.conv2(out)))
        out = F.relu(self.bn3(self.conv3(out)))
        out = F.relu(self.bn4(self.conv4(out)))
        out = F.relu(self.bn5(self.conv5(out)))
        return out


class KSImplicit(nn.Module):
    """u_t = -u_xx - u_xxxx discretised with the fixed 5-point stencil of imex.py:20-36 (requires_grad=False)."""

    def __init__(self, dx, dtype=torch.float64):
        super().__init__()
        self.A = nn.Conv1d(1, 1, kernel_size=5, padding="same", padding_mode="circular", bias=False)
        # the reference builds the stencil with torch.tensor(<python floats>) -- float32 -- and only then calls .double()
        # (imex.py:20-36, KS.py:470): in a double-precision run the coefficients are the float32-ROUNDED values (pinned by
        # tests/golden/ks_ref_fp64.pt)
        K = torch.tensor([[[-1.0 / dx ** 4, 4.0 / dx ** 4 - 1.0 / dx ** 2, -6.0 / dx ** 4 + 2.0 / dx ** 2,
                            4.0 / dx ** 4 - 1.0 / dx ** 2, -1.0 / dx ** 4]]], dtype=torch.float32).to(dtype)
        self.A.weight = nn.Parameter(K, requires_grad=False)
        self.nfe = 0

    def forward(self, t, y):
        self.nfe += 1
        return torch.squeeze(self.A(torch.unsqueeze(y, 1)), 1)


class KSExplicit(nn.Module):
    def __init__(self, n, hidden=None, dtype=torch.float64, seed=0):
        super().__init__()
        hidden = hidden or n * 25 // 8
        torch.manual_seed(seed)
        self.F = nn.Sequential(nn.Linear(n, hidden), nn.ReLU(), nn.Linear(hidden, hidden), nn.ReLU(),
                               nn.Linear(hidden, hidden), nn.ReLU(), nn.Linear(hidden, hidden), nn.ReLU(),
                               nn.Linear(hidden, n))
        for m in self.F.modules():
            if isinstance(m, nn.Linear):
                nn.init.normal_(m.weight, mean=0, std=0.01)
        self.to(dtype)
        self.nfe = 0

    def forward(self, t, y):
        self.nfe += 1
        return -self.F(y)


def ks_dx(n):
    return 22.0 / n


class BurgersImplicit(nn.Module):
    """Viscous term alpha u_xx on a periodic grid: the fixed 3-point stencil of examples-sinode/Burgers/Burgers.py:163-195
    (built in float32 like the reference, then cast)."""

    def __init__(self, n, alpha=8e-4, dtype=torch.float64):
        super().__init__()
        dx = 1.0 / n
        self.A = nn.Conv1d(1, 1, kernel_size=3, padding="same", padding_mode="circular", bias=False)
        K = torch.tensor([[[alpha / dx ** 2, -2.0 * alpha / dx ** 2, alpha / dx ** 2]]], dtype=torch.float32).to(dtype)
        self.A.weight = nn.Parameter(K, requires_grad=False)
        self.nfe = 0

    def forward(self, t, y):
        self.nfe += 1
        return torch.squeeze(self.A(torch.unsqueeze(y, 1)), 1)


class BurgersExplicit(nn.Module):
    """Burgers.py:134-160: five Linear layers of width 9N/8 with ReLU, weights N(0, 0.1^2), zero biases, returning +net(y)."""

    def __init__(self, n, dtype=torch.float64, seed=0):
        super().__init__()
        torch.manual_seed(seed)
        h = n * 9 // 8
        self.net = nn.Sequential(nn.Linear(n, h), nn.ReLU(), nn.Linear(h, h), nn.ReLU(), nn.Linear(h, h), nn.ReLU(),
                                 nn.Linear(h, h), nn.ReLU(), nn.Linear(h, n))
        for m in self.net.modules():
            if isinstance(m, nn.Linear):
                nn.init.normal_(m.weight, mean=0, std=0.1)
                nn.init.constant_(m.bias, val=0)
        self.to(dtype)
        self.nfe = 0

    def forward(self, t, y):
        self.nfe += 1
        return self.net(y)
