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


def forward(layers, z, e, tau, abs_terms=False):
    """F = (f, -div) flattened like FlattenFunc, and what the adjoint needs per layer.  With abs_terms, also the sum of the
    absolute values of the terms of the last layer's sums (the scale of each entry's rounding error)."""
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
    F = torch.cat((a.reshape(-1), -div))
    if not abs_terms:
        return F, cache
    aW = W.abs()
    f_abs = gam.abs() * (x.abs() @ aW.T + b.abs()) + c.abs()
    div_abs = (e.abs() * gam.abs() * (v.abs() @ aW.T)).sum(1)
    return F, cache, torch.cat((f_abs.reshape(-1), div_abs))


def vjp(layers, cache, e, w, tau, abs_terms=False):
    """(J^T w flattened, [[dW, db, dhbw, dhgw, dhgb] per layer]) for the cotangent w = (w_z, w_logp).

    With abs_terms, also the same two results with the operands of every product and every sum in absolute value -- for
    example |Pbar|^T |x| + |Qbar|^T |v| for dW and sum |Pbar| for db -- the scale against which each entry's rounding error
    is measured."""
    B, D = e.shape
    wz, wl = w[:B * D].view(B, D), w[B * D:]
    abar, ubar = wz, -wl[:, None] * e
    grads = [None] * len(layers)
    if abs_terms:
        abar_a, ubar_a = abar.abs(), ubar.abs()
        grads_a = [None] * len(layers)
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
        W = m._layer.weight
        xb, vb = Pb @ W, Qb @ W
        if abs_terms:
            g_a, aW = gam.abs(), W.abs()
            Pa, Qa = g_a * abar_a, g_a * ubar_a
            gg_a = (abar_a * k["P"].abs() + ubar_a * k["Q"].abs()).sum(0) * g_a * (1 - gam).abs()
            grads_a[l] = [Pa.T @ k["x"].abs() + Qa.T @ k["v"].abs(), Pa.sum(0), (abar_a.sum(0) * abs(tau))[:, None],
                          (gg_a * abs(tau))[:, None], gg_a]
            xb_a, vb_a = Pa @ aW, Qa @ aW
        if l > 0:
            s, u = cache[l - 1]["s"], cache[l - 1]["u"]
            abar, ubar = s * xb + s * (1 - s) * u * vb, s * vb
            if abs_terms:
                abar_a, ubar_a = s * xb_a + s * (1 - s) * u.abs() * vb_a, s * vb_a
    zeros = torch.zeros(B, dtype=w.dtype, device=w.device)
    jtw = torch.cat((xb.reshape(-1), zeros))
    if not abs_terms:
        return jtw, grads
    return jtw, grads, torch.cat((xb_a.reshape(-1), zeros)), grads_a
