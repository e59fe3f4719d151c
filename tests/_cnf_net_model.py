"""Host model of csrc/cnf_net.cu: the FFJORD ConcatSquash network of any depth, its Hutchinson trace as the forward tangent
of the probe, and the adjoint stage in closed form (J^T w and the five parameter gradients of every layer), restated in
torch on whatever device and dtype the inputs have.  Notation of the kernel file (row vectors, x_0 = z, v_0 = e)."""
import torch


def gates(layers, tau):
    """[(gamma_l, c_l)] at the (already rounded) time tau."""
    out = []
    for m in layers:
        hgw, hgb, hbw = m._hyper_gate.weight[:, 0], m._hyper_gate.bias, m._hyper_bias.weight[:, 0]
        out.append((torch.sigmoid(hgw * tau + hgb), hbw * tau))
    return out


def _softplus_sigmoid(a):
    """torch.nn.Softplus(beta=1, threshold=20) and its derivative: identity with slope exactly 1 above the threshold."""
    above = a > 20
    sp = torch.where(above, a, torch.log1p(torch.exp(torch.where(above, torch.zeros_like(a), a))))
    s = torch.where(above, torch.ones_like(a), torch.sigmoid(a))
    return sp, s


def forward(layers, z, e, tau):
    """F = (f, -div) flattened like FlattenFunc, and what the adjoint needs per layer."""
    gs = gates(layers, tau)
    x, v = z, e
    cache = []
    for l, (m, (gam, c)) in enumerate(zip(layers, gs)):
        W, b = m._layer.weight, m._layer.bias
        P = x @ W.T + b
        Q = v @ W.T
        a = gam * P + c
        u = gam * Q
        sp, s = _softplus_sigmoid(a)
        cache.append(dict(x=x, v=v, P=P, Q=Q, u=u, s=s, gam=gam))
        if l < len(layers) - 1:
            x, v = sp, s * u
    div = (e * u).sum(1)
    return torch.cat((a.reshape(-1), -div)), cache


def vjp(layers, cache, e, w, tau):
    """(J^T w flattened, [[dW, db, dhbw, dhgw, dhgb] per layer]) for the cotangent w = (w_z, w_logp)."""
    B, D = e.shape
    wz, wl = w[:B * D].view(B, D), w[B * D:]
    abar, ubar = wz, -wl[:, None] * e
    grads = [None] * len(layers)
    for l in range(len(layers) - 1, -1, -1):
        k, m = cache[l], layers[l]
        gam = k["gam"]
        Pb, Qb = gam * abar, gam * ubar
        dW = Pb.T @ k["x"] + Qb.T @ k["v"]
        db = Pb.sum(0)
        gbar = (abar * k["P"] + ubar * k["Q"]).sum(0)
        cbar = abar.sum(0)
        gg = gbar * gam * (1 - gam)
        grads[l] = [dW, db, (cbar * tau)[:, None], (gg * tau)[:, None], gg]
        xb, vb = Pb @ m._layer.weight, Qb @ m._layer.weight
        if l > 0:
            s, u = cache[l - 1]["s"], cache[l - 1]["u"]
            abar, ubar = s * xb + s * (1 - s) * u * vb, s * vb
    return torch.cat((xb.reshape(-1), torch.zeros(B, dtype=w.dtype, device=w.device))), grads
