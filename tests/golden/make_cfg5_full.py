"""Generates tests/golden/cfg5_full_fp64.pt: BASELINE config 5 at FULL size (KS N=1024, MLP hidden 3200, batch 256, fp64,
ARKIMEX type 3, h = 0.2, one step, -snes_type ksponly, linear_solver='torch') through the CPU ORACLE on seeded inputs.
Run once in the build container (about a minute on 8 cores):   python tests/golden/make_cfg5_full.py
Stored (under 1 MB): final state and lambda as 32 sampled batch rows in full + sum / abs-sum / norm of the whole arrays, mu
(37.3 M entries) as 4096 sampled entries + sum / abs-sum / norm."""
import os
import sys
import time

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import OracleODEPetsc  # noqa: E402
from _workloads import KSExplicit, KSImplicit, ks_dx  # noqa: E402


def main():
    N, H, B, seed = 1024, 3200, 256, 4
    torch.set_num_threads(os.cpu_count())
    g = torch.Generator().manual_seed(seed)
    u0 = 0.5 * torch.randn(B, N, generator=g, dtype=torch.float64)
    gout = torch.randn(2, B, N, generator=g, dtype=torch.float64)
    t = torch.tensor([0.0, 0.2], dtype=torch.float64)
    argv = ["-ts_adapt_type", "none", "-snes_type", "ksponly", "-ts_arkimex_type", "3"]
    f_im, f_ex = KSImplicit(ks_dx(N)), KSExplicit(N, hidden=H)
    ode = OracleODEPetsc(argv)
    ode.setupTS(u0, f_im, step_size=0.2, method="imex", imex_form=True, func2=f_ex, batch_size=B, linear_solver="torch")
    t0 = time.time()
    y0 = u0.clone().requires_grad_(True)
    out = ode.odeint_adjoint(y0, t)
    (out * gout).sum().backward()
    mu = torch.cat([p.grad.reshape(-1) for p in f_ex.parameters()])
    print("oracle pass: %.1f s, np = %d" % (time.time() - t0, mu.numel()))
    gi = torch.Generator().manual_seed(99)
    idx = torch.randint(0, mu.numel(), (4096,), generator=gi)
    rows = torch.randperm(B, generator=gi)[:32].sort().values
    fx = {"N": N, "H": H, "B": B, "seed": seed, "rows": rows, "mu_index": idx, "mu_sample": mu[idx].clone(),
          "mu_sum": float(mu.sum()), "mu_abs_sum": float(mu.abs().sum()), "mu_norm": float(mu.norm())}
    for name, x in (("u", out[-1].detach()), ("lam", y0.grad)):
        fx.update({name + "_rows": x[rows].clone(), name + "_sum": float(x.sum()), name + "_abs_sum": float(x.abs().sum()),
                   name + "_norm": float(x.norm())})
    torch.save(fx, os.path.join(HERE, "cfg5_full_fp64.pt"))


if __name__ == "__main__":
    main()
