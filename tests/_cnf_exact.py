"""FFJORD modules with the exact trace, and a host model of what csrc/cnf_net.cu evaluates for them.

  * divergence_bf  -- ffjord-pnode/lib/layers/odefunc.py:21-26: the exact trace of df/dz, one autograd call per state
                      component, summed in component order
  * ODEfuncEvalBF  -- ODEfunc.forward of odefunc.py:345-385 with its eval-mode branch: a 2-D state in eval mode takes
                      divergence_bf whatever divergence_fn says
  * exact_cnf      -- _workloads.CNFFunc with divergence_fn = divergence_bf
  * forward / vjp  -- the exact-trace forward and adjoint stage in closed form, D tangent chains v_0^(k) = e_k (notation of
                      the header of csrc/cnf_net.cu and of _cnf_net_model, which holds the Hutchinson case)
"""
import torch

import _cnf_net_model as hmodel
from _workloads import ODEfunc, ODEnet, FlattenFunc, CNFFunc


def divergence_bf(dx, y, **unused_kwargs):
    sum_diag = 0.0
    for i in range(y.shape[1]):
        sum_diag += torch.autograd.grad(dx[:, i].sum(), y, create_graph=True)[0].contiguous()[:, i].contiguous()
    return sum_diag.contiguous()


class ODEfuncEvalBF(ODEfunc):
    """ODEfunc whose eval mode takes the exact trace for 2-D states (odefunc.py:372-375)."""

    def forward(self, t, states):
        y = states[0]
        self._num_evals += 1
        t = torch.tensor(t).type_as(y)
        if self._e is None:
            self._e = torch.randn_like(y)
        with torch.set_grad_enabled(True):
            y.requires_grad_(True)
            dy = self.diffeq(t, y)
            if not self.training and dy.view(dy.shape[0], -1).shape[1] == 2:
                divergence = divergence_bf(dy, y).view(y.shape[0], 1)
            else:
                divergence = self.divergence_fn(dy, y, e=self._e).view(y.shape[0], 1)
        return (dy, -divergence)


def exact_cnf(batch, dim, hidden_dims, dtype=torch.float64, seed=0, t_via_f32=True):
    func = CNFFunc(batch, dim, hidden_dims, dtype=dtype, seed=seed, t_via_f32=t_via_f32)
    func.base_func.divergence_fn = divergence_bf
    return func


def eval_branch_cnf(batch, hidden_dims, dtype=torch.float64, seed=0):
    """A D = 2 FFJORD module with the Hutchinson divergence_fn and the eval-mode branch to the exact trace."""
    torch.manual_seed(seed)
    odefunc = ODEfuncEvalBF(ODEnet(hidden_dims, 2).to(dtype))
    g = torch.Generator().manual_seed(seed + 1)
    odefunc._e = torch.randn(batch, 2, generator=g, dtype=torch.float64).to(dtype)
    y0 = (torch.zeros(batch, 2, dtype=dtype), torch.zeros(batch, 1, dtype=dtype))
    return FlattenFunc(odefunc, y0)


def forward(layers, z, tau):
    """F = (f, -tr J) flattened like FlattenFunc, and what the adjoint needs per layer; tangents are [D, B, width]."""
    B, D = z.shape
    x = z
    v = torch.eye(D, dtype=z.dtype, device=z.device)[:, None, :].expand(D, B, D)
    cache = []
    for l, (m, (gam, c)) in enumerate(zip(layers, hmodel.gates(layers, tau))):
        W, b = m._layer.weight, m._layer.bias
        P = x @ W.T + b
        Q = v @ W.T
        a = gam * P + c
        u = gam * Q
        sp, s = hmodel._softplus_sigmoid(a)
        cache.append(dict(x=x, v=v, P=P, Q=Q, u=u, s=s, gam=gam))
        if l < len(layers) - 1:
            x, v = sp, s * u
    div = sum(u[k, :, k] for k in range(D))
    return torch.cat((a.reshape(-1), -div)), cache


def vjp(layers, cache, w, tau):
    """(J^T w flattened, [[dW, db, dhbw, dhgw, dhgb] per layer]) for the cotangent w = (w_z, w_logp)."""
    D = layers[0]._layer.in_features
    B = w.numel() // (D + 1)
    wz, wl = w[:B * D].view(B, D), w[B * D:]
    abar = wz
    ubar = torch.zeros(D, B, D, dtype=w.dtype, device=w.device)
    for k in range(D):
        ubar[k, :, k] = -wl
    grads = [None] * len(layers)
    for l in range(len(layers) - 1, -1, -1):
        k, m = cache[l], layers[l]
        gam = k["gam"]
        Pb, Qb = gam * abar, gam * ubar
        dW = Pb.T @ k["x"] + (Qb.transpose(1, 2) @ k["v"]).sum(0)
        db = Pb.sum(0)
        gbar = (abar * k["P"]).sum(0) + (ubar * k["Q"]).sum((0, 1))
        cbar = abar.sum(0)
        gg = gbar * gam * (1 - gam)
        grads[l] = [dW, db, (cbar * tau)[:, None], (gg * tau)[:, None], gg]
        W = m._layer.weight
        xb, vb = Pb @ W, Qb @ W
        if l > 0:
            s, u = cache[l - 1]["s"], cache[l - 1]["u"]
            abar, ubar = s * xb + s * (1 - s) * (u * vb).sum(0), s * vb
    jtw = torch.cat((xb.reshape(-1), torch.zeros(B, dtype=w.dtype, device=w.device)))
    return jtw, grads
