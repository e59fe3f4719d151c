"""Per-unit parity of both FFJORD evaluators (the fused sweeps of csrc/cnf_rk.cu and the evaluator of any depth in
csrc/cnf_net.cu) where their arithmetic branches or is least accurate: units above, just below and far above torch's
softplus threshold (a = 20), units deep in the negative tail, gates in their tails, and both ways a module may round t.

Every hidden unit is placed in one of six regimes by j mod 6, so every regime sits in every chunk of hidden units of the
fused adjoint (2 x 30 units in fp64, 4 x 15 in fp32) and the units on either side of each chunk boundary are in different
regimes.  A unit is placed by its bias, with its weight row and the weight column that reads it scaled down so that the flow
stays mild; the unit's own gradient scales with it, so per-unit relative checks are unaffected.

* One Euler step from t = 0.3 (not representable in fp32) is a closed form of one evaluation of the host model
  (tests/_cnf_net_model.py): u1 = u0 + h F, lambda0 = g0 + g1 + h J^T g1, mu = h (dF/dtheta)^T g1.  Every entry is held to
  tol x (its sum of absolute terms), failures reported per (parameter, unit); in fp64 each unit also to its own norm.
* RK4 and adaptive dopri5 against the oracle: trajectory, lambda and each parameter tensor at the bars of test_gpu_cnf.py,
  and each unit's weight row, bias entry and gate entries against the norm of those five gradients of the unit together,
  and the weight column that reads it against its own norm.

Two roundings are inherent in the arithmetic and are allowed on top of the tolerance:
  * g (1 - g) of a gate near 1 carries the rounding of g divided by 1 - g: 4 units of roundoff of g over 1 - g (7e-11 in
    fp64 at |x| = 12, a few percent in fp32).  Gate arguments stay within |x| <= 12: beyond about 16 the fp64 rounding of
    g alone moves g (1 - g) by more than 1e-10, and two correct implementations would disagree.
  * The fused fp32 softplus, log(1 + e^a) with 1 + e^a rounded to fp32, is exact to one unit of roundoff absolutely, not
    relatively: the weight gradient that reads a unit far below zero is held to that.
"""
import copy
import gc
import weakref

import pytest
import torch

import _cnf_net_model as model
from oracle import OracleODEPetsc
from pnode_b200.options import Options
from _problems import rel_err
from _workloads import CNFFunc, cnf_to

pytestmark = pytest.mark.gpu

REGIMES = ("stock", "above", "below", "far", "negative", "gate")
BANDS = {"stock": (-25.0, 18.0), "above": (20.2, 21.8), "below": (18.2, 19.8), "far": (30.0, 45.0),
         "negative": (-45.0, -25.0), "gate": (-25.0, 18.0)}
TOL = {torch.float64: 1e-10, torch.float32: 1e-4}
ROUNDOFF = {torch.float64: 2.0 ** -53, torch.float32: 2.0 ** -24}
GATE_OUT = (1, 4)  # output dimensions of the last layer with their gate in its tail
NAMES = ("W", "b", "hbw", "hgw", "hgb")
FUSED, NET = "fused-cnf-rk", "generic+cnf-net-rhs"


def regime(j):
    return REGIMES[j % 6]


def _gate_tail(m, j, k):
    """|hgw t + hgb| in [10.5, 11.8] for t in [0, 1.3], the sign alternating with k."""
    sign = 1.0 if k % 2 == 0 else -1.0
    m._hyper_gate.weight[j, 0] = sign
    m._hyper_gate.bias[j] = 10.5 * sign


def tail_model(B, D, hidden, t_via_f32, seed):
    """CNFFunc in fp64 with every hidden unit of every layer placed in its regime (j mod 6)."""
    func = CNFFunc(B, D, hidden, dtype=torch.float64, seed=seed, t_via_f32=t_via_f32)
    layers = list(func.base_func.diffeq.layers)
    g = torch.Generator().manual_seed(seed + 100)
    with torch.no_grad():
        for l, (m, nxt) in enumerate(zip(layers[:-1], layers[1:])):
            for j in range(m._layer.out_features):
                r = regime(j)
                if r == "stock":
                    continue
                if r == "gate":
                    _gate_tail(m, j, j // 6)
                    continue
                lo, hi = BANDS[r]
                target = lo + (hi - lo) * (0.3 + 0.4 * float(torch.rand(1, generator=g, dtype=torch.float64)))
                m._hyper_gate.weight[j] = 0.0  # gate and shift constant in t: a stays in its band along the flow
                m._hyper_bias.weight[j] = 0.0
                m._layer.weight[j] *= 0.02
                m._layer.bias[j] = target / torch.sigmoid(m._hyper_gate.bias[j])
                nxt._layer.weight[:, j] *= 0.05
        for k, j in enumerate(GATE_OUT):
            _gate_tail(layers[-1], j, k)
    return func


def as_dtype(func, dtype):
    f = copy.deepcopy(func).to(dtype)
    f.base_func._e = f.base_func._e.to(dtype)
    f.y0 = tuple(x.to(dtype) for x in f.y0)
    return f


def inputs(B, D, T, dtype, seed=2):
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(B, D, generator=g, dtype=torch.float64)
    u0 = torch.cat((z.view(-1), torch.zeros(B, dtype=torch.float64))).to(dtype)
    gout = torch.randn(T, B * (D + 1), generator=g, dtype=torch.float64).to(dtype)
    return u0, gout


def tau_of(t, via_f32, dtype):
    """The time the kernels evaluate at: rounded through fp32 by the reference's module, and in any fp32 run."""
    return float(torch.tensor(t, dtype=torch.float32)) if (via_f32 or dtype == torch.float32) else t


def assert_bands(func, z, tau):
    """Every (trajectory, unit) pair of every hidden layer lies in its regime's band at state z."""
    layers = list(func.base_func.diffeq.layers)
    with torch.no_grad():
        _, cache = model.forward(layers, z.double(), func.base_func._e.double(), tau)
        gs = model.gates(layers, tau)
    for l in range(len(layers) - 1):
        a = cache[l]["gam"] * cache[l]["P"] + gs[l][1]
        for j in range(a.shape[1]):
            lo, hi = BANDS[regime(j)]
            assert bool((a[:, j] > lo).all() and (a[:, j] < hi).all()), \
                "layer %d unit %d (%s): a in [%.3f, %.3f]" % (l, j, regime(j), float(a[:, j].min()), float(a[:, j].max()))
            assert float((a[:, j] - 20).abs().min()) >= 0.2
    for l, (gam, _) in enumerate(gs):
        x = torch.logit(gam)
        for j in range(gam.shape[0]):
            tail = (l < len(layers) - 1 and regime(j) == "gate") or (l == len(layers) - 1 and j in GATE_OUT)
            assert float(x[j].abs()) <= 12.0 and (not tail or float(x[j].abs()) >= 10.0), (l, j, float(x[j]))


def run_gpu(func, u0, t, gout, method, step, argv):
    from pnode import petsc_adjoint

    Options.clear_all()
    Options.insert_args(argv)
    f = cnf_to(copy.deepcopy(func), "cuda")
    ode = petsc_adjoint.ODEPetsc()
    ode.setupTS(u0.cuda(), f, step_size=step, method=method, enable_adjoint=True)
    y0 = u0.cuda().clone().requires_grad_(True)
    out = ode.odeint_adjoint(y0, t.cuda())
    (out * gout.cuda()).sum().backward()
    torch.cuda.synchronize()
    return out.detach().cpu(), y0.grad.cpu(), [p.grad.cpu() for p in f.parameters()], ode


def run_oracle(func, u0, t, gout, method, step, argv):
    Options.clear_all()
    Options.insert_args(argv)
    f = copy.deepcopy(func)
    ode = OracleODEPetsc(argv)
    ode.setupTS(u0, f, step_size=step, method=method, enable_adjoint=True)
    y0 = u0.clone().requires_grad_(True)
    out = ode.odeint_adjoint(y0, t)
    (out * gout).sum().backward()
    return out.detach(), y0.grad, [p.grad for p in f.parameters()], ode


def spec_of(ode):
    return ode._fused.spec if ode.path == FUSED else ode._cb_ex.spec


def gate_floor(gam, dtype):
    """Relative error of g (1 - g) that the rounding of g alone can cause: 4 units of roundoff of g over 1 - g."""
    return 4.0 * ROUNDOFF[dtype] * gam / (1.0 - gam)


# ---------------------------------------------------------------------------------------------------------------------
# one Euler step against the host model, entry by entry

def euler_reference(func, u0, gout, t0, h, tau):
    """(u1, lambda0, [mu per parameter]) of one Euler step, each as (value, sum of absolute terms), and the gates."""
    bf = func.base_func
    layers = list(bf.diffeq.layers)
    e = bf._e
    B, D = e.shape
    with torch.no_grad():
        F, cache, F_a = model.forward(layers, u0[:B * D].view(B, D), e, tau, abs_terms=True)
        jtw, grads, jtw_a, grads_a = model.vjp(layers, cache, e, gout[1], tau, abs_terms=True)
    u1 = (u0 + h * F, u0.abs() + h * F_a)
    lam = (gout[0] + gout[1] + h * jtw, gout[0].abs() + gout[1].abs() + h * jtw_a)
    mu = [(h * g, h * ga) for gl, gla in zip(grads, grads_a) for g, ga in zip(gl, gla)]
    return u1, lam, mu, [c["gam"] for c in cache]


def entry_failures(what, got, ref, S, bar):
    """Entries with |got - ref| > bar, the worst per row (= per unit for the parameters)."""
    n = ref.shape[0]
    got, ref, S, bar = got.double().reshape(n, -1), ref.reshape(n, -1), S.reshape(n, -1), bar.reshape(n, -1)
    ratio = (got - ref).abs() / torch.where(bar > 0, bar, torch.full_like(bar, 1e-300))
    out = []
    for j in torch.nonzero((ratio > 1).any(1)).reshape(-1).tolist():
        w = int(ratio[j].argmax())
        out.append("%s[%d]: %.3g x bar (err %.3g, S %.3g)" % (what, j, float(ratio[j, w]), float((got[j, w] - ref[j, w]).abs()),
                                                           float(S[j, w])))
    return out


SINGLE = [pytest.param(FUSED, 6, (60,), 77, id="fused-B77"), pytest.param(FUSED, 6, (60,), 20001, id="fused-B20001"),
          pytest.param(NET, 6, (37, 129), 77, id="net-B77"), pytest.param(NET, 6, (37, 129), 300, id="net-B300")]


@pytest.mark.parametrize("via_f32", [True, False], ids=["t-f32", "t-f64"])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("path,D,hidden,B", SINGLE)
def test_one_euler_step_every_entry(path, D, hidden, B, dtype, via_f32):
    t0 = 0.3
    func = as_dtype(tail_model(B, D, hidden, via_f32, seed=B + len(hidden)), dtype)
    u0, gout = inputs(B, D, 2, dtype)
    t = torch.tensor([t0, 0.8], dtype=torch.float64)
    p = run_gpu(func, u0, t, gout, "euler", 0.5, [])
    ode = p[3]
    assert ode.path == path
    assert spec_of(ode).t_via_f32 == (1 if via_f32 or dtype == torch.float32 else 0)
    assert len(ode._loop.attempts) == 1
    h = ode._loop.attempts[0][1]
    assert h == pytest.approx(0.5, abs=1e-15)

    ref64 = as_dtype(func, torch.float64)  # the host model on the inputs the kernels received
    tau = tau_of(t0, via_f32, dtype)
    assert_bands(ref64, u0.double()[:B * D].view(B, D), tau)
    (u1, u1_a), (lam, lam_a), mu, gams = euler_reference(ref64, u0.double(), gout.double(), t0, h, tau)
    tol = TOL[dtype]
    bad = entry_failures("u1", p[0][1], u1, u1_a, tol * u1_a) + entry_failures("lambda0", p[1], lam, lam_a, tol * lam_a)
    assert len(p[2]) == len(mu) == 5 * (len(hidden) + 1)
    for i, (got, (ref, S)) in enumerate(zip(p[2], mu)):
        l, name = i // 5, NAMES[i % 5]
        bar = tol * S
        if name in ("hgw", "hgb"):
            bar = bar + gate_floor(gams[l], dtype)[:, None].reshape(S.shape) * S
        if name == "W" and l > 0 and dtype == torch.float32:
            # the fused fp32 softplus, log(1 + e^a) with 1 + e^a rounded, is exact to one unit of roundoff absolutely
            # (csrc/cnf_rk.cu): the weight gradient reading it is known to that times sum |Pbar| = the bias gradient's S
            bar = bar + ROUNDOFF[dtype] * mu[5 * l + 1][1][:, None]
        bad += entry_failures("layer %d %s" % (l, name), got, ref, S, bar)
    # A wrong slope scales every term of a unit's sums alike, and the sums over the batch cancel: against the sum of
    # absolute terms such an error shrinks like 1/sqrt(B).  In fp64 each unit is also held to its own norm; in fp32 that
    # norm can sit below the rounding of a sum over 20001 trajectories.
    if dtype == torch.float64:
        bad += unit_failures(p[2], [m[0] for m in mu], hidden, tol, [gate_floor(g, dtype).tolist() for g in gams])
    assert not bad, "%d failures: %s" % (len(bad), "; ".join(bad[:40]))


# ---------------------------------------------------------------------------------------------------------------------
# several steps against the oracle, unit by unit

def unit_failures(got, ref, hidden, tol, gate_rel):
    """Each hidden unit's weight row, bias entry and gate entries, and each output's entries of the last layer, held to
    tol times the norm of that unit's five gradients together (gate entries with the rounding of g on top); the weight
    column that reads a hidden unit, to its own norm.  Deep-negative units are left to the single-step test: their own
    norm can be dominated by cancellation."""
    bad = []
    L = len(hidden) + 1
    for l in range(L):
        for j in range(got[5 * l].shape[0]):
            if l < L - 1 and regime(j) == "negative":
                continue
            own = [(NAMES[i] if i else "W row", got[5 * l + i][j], ref[5 * l + i][j]) for i in range(5)]
            den = float(torch.cat([r.double().reshape(-1) for _, _, r in own]).norm())
            checks = [(name, a, r, den) for name, a, r in own]
            if l < L - 1:
                col = ref[5 * l + 5][:, j]
                checks.append(("reading W column", got[5 * l + 5][:, j], col, float(col.double().norm())))
            for name, a, r, d in checks:
                err = float((a.double() - r.double()).norm())
                bar = tol * d + (gate_rel[l][j] * float(r.double().norm()) if name in ("hgw", "hgb") else 0.0)
                if not err <= bar:
                    bad.append("layer %d unit %d (%s) %s: %.3g" % (l, j, regime(j) if l < L - 1 else "out", name, err / d))
    return bad


MULTI = [pytest.param(FUSED, (60,), id="fused"), pytest.param(NET, (37, 129), id="net")]


@pytest.mark.parametrize("method", ["rk4", "dopri5"])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("path,hidden", MULTI)
def test_several_steps_every_unit_against_the_oracle(path, hidden, dtype, method):
    B, D = 77, 6
    via_f32 = method == "rk4"  # the reference's module under RK4, the t-f64 module under dopri5
    func = as_dtype(tail_model(B, D, hidden, via_f32, seed=7 + len(hidden)), dtype)
    u0, gout = inputs(B, D, 2, dtype, seed=5)
    t = torch.tensor([0.3, 1.3], dtype=torch.float64)
    if method == "rk4":
        argv, step = ["-ts_adapt_type", "none"], 0.25
    else:
        tt = "1e-6" if dtype == torch.float64 else "1e-4"
        argv, step = ["-ts_rtol", tt, "-ts_atol", tt], 0.05
    o = run_oracle(func, u0, t, gout, method, step, argv)
    p = run_gpu(func, u0, t, gout, method, step, argv)
    assert p[3].path == path
    if method == "dopri5":
        lo, lp = o[3].ts.log, p[3]._loop.attempts
        assert [a[2] for a in lo] == [a[2] for a in lp], "accept/reject pattern"
        for a, b in zip(lo, lp):
            assert a[1] == pytest.approx(b[1], rel=1e-8 if dtype == torch.float64 else 2e-2)
    else:
        assert p[3]._loop.steps == 4

    ref64 = as_dtype(func, torch.float64)
    for tv, z in ((0.3, u0), (1.3, o[0][-1])):
        assert_bands(ref64, z.double()[:B * D].view(B, D), tau_of(tv, via_f32, dtype))
    tol = TOL[dtype]
    assert rel_err(p[0], o[0]) < tol, ("trajectory", rel_err(p[0], o[0]))
    assert rel_err(p[1], o[1]) < tol, ("lambda", rel_err(p[1], o[1]))
    for i, (a, b) in enumerate(zip(p[2], o[2])):
        assert rel_err(a, b) < tol, ("layer %d %s" % (i // 5, NAMES[i % 5]), rel_err(a, b))
    gate_rel = []
    for tv in (0.3, 1.3):
        gs = model.gates(list(ref64.base_func.diffeq.layers), tau_of(tv, via_f32, dtype))
        fl = [gate_floor(g, dtype) for g, _ in gs]
        gate_rel = fl if not gate_rel else [torch.maximum(x, y) for x, y in zip(gate_rel, fl)]
    bad = unit_failures(p[2], [g.cpu() for g in o[2]], hidden, tol, [x.tolist() for x in gate_rel])
    assert not bad, "%d failures: %s" % (len(bad), "; ".join(bad[:40]))


# ---------------------------------------------------------------------------------------------------------------------
# the recogniser's verdict lives as long as the module

def test_recognised_verdict_dies_with_the_module():
    from pnode_b200 import fused

    B, D = 16, 6
    meta = torch.empty(B * (D + 1), dtype=torch.float64, device="cuda")
    gc.collect()  # entries of modules freed by earlier tests go now, not in the middle of this one
    f32 = cnf_to(CNFFunc(B, D, (60,), dtype=torch.float64, seed=1), "cuda")
    spec = fused.recognise_cnf(f32, meta)
    assert spec is not None and spec.t_via_f32 == 1
    n = len(fused._CNF_RECOGNISED)
    ref = weakref.ref(f32.base_func)
    del f32, spec
    gc.collect()
    assert ref() is None
    assert len(fused._CNF_RECOGNISED) == n - 1
    # a module that keeps t in fp64, possibly at the freed module's addresses, gets a verdict of its own
    f64 = cnf_to(CNFFunc(B, D, (60,), dtype=torch.float64, seed=1, t_via_f32=False), "cuda")
    spec = fused.recognise_cnf(f64, meta)
    assert spec is not None and spec.t_via_f32 == 0
