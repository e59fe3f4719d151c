"""Fused-kernel paths: recognisers that map a user `nn.Module` onto a hand-written sweep kernel, and the host glue
that launches it.  A module that is not recognised (or `-pnode_fused 0`) runs on the generic path of engine.py -- both
execute on the GPU; neither is a fallback for a missing library.

Currently fused: tiny-state MLPs  f(t,y) = Linear(H,d)(tanh(Linear(d,H)(phi(y)))), phi = y**3 | y  -- the spiral model of
examples-pnode/ode_demo_petsc.py:207-230 -- under any fixed-step explicit RK scheme (csrc/mlp_rk.cu).
"""
import ctypes as C
import weakref

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from .controller import fixed_schedule
from .device import _stream, dtype_code
from .errors import Error

_STEP_DTYPE = np.dtype([("t", "<f8"), ("h", "<f8"), ("out_slot", "<i4"), ("in_slot", "<i4")])
assert _STEP_DTYPE.itemsize == C.sizeof(_lib.Step)


class MlpSpec:
    def __init__(self, lin1, lin2, phi, dim, hidden):
        self.lin1, self.lin2, self.phi, self.dim, self.hidden = lin1, lin2, phi, dim, hidden

    def params(self):
        return [self.lin1.weight, self.lin1.bias, self.lin2.weight, self.lin2.bias]


def recognise_mlp(func, u_meta):
    """Return an MlpSpec when `func(t, y)` is provably  lin2(tanh(lin1(phi(y))))  acting on the last axis of y:
    structural match of the module tree AND a numerical probe of the forward on random inputs at two times."""
    if not isinstance(func, nn.Module) or not u_meta.is_cuda or u_meta.dim() < 1:
        return None
    mods = [m for m in func.modules() if m is not func and not isinstance(m, (nn.Sequential, nn.ModuleList))]
    lins = [m for m in mods if isinstance(m, nn.Linear)]
    tanhs = [m for m in mods if isinstance(m, nn.Tanh)]
    if len(lins) != 2 or len(tanhs) != 1 or len(mods) != 3:
        return None
    lin1, lin2 = lins
    d = u_meta.shape[-1]
    if lin1.bias is None or lin2.bias is None:
        return None
    if lin1.in_features != d or lin2.out_features != d or lin1.out_features != lin2.in_features:
        return None
    plist = [p for p in func.parameters() if p.requires_grad]
    want = [lin1.weight, lin1.bias, lin2.weight, lin2.bias]
    if len(plist) != 4 or any(a is not b for a, b in zip(plist, want)):
        return None
    if any(p.dtype != u_meta.dtype or p.device != u_meta.device or not p.is_contiguous() for p in want):
        return None
    if len(list(func.buffers())) != 0:
        return None
    # numerical probe (a handful of tiny launches, once per func identity)
    with torch.no_grad():
        g = torch.Generator(device="cpu").manual_seed(1234)
        shape = (3,) + tuple(u_meta.shape[1:]) if u_meta.dim() > 1 else tuple(u_meta.shape)
        x = (torch.rand(shape, generator=g, dtype=torch.float64) * 2 - 1).to(device=u_meta.device, dtype=u_meta.dtype)
        try:
            y0 = func(0.0, x)
            y1 = func(0.73, x)
        except Exception:
            return None
        if y0.shape != x.shape or not torch.equal(y0, y1):
            return None
        tol = 1e-5 if u_meta.dtype == torch.float32 else 1e-12
        for phi, fn in ((1, lambda v: v ** 3), (0, lambda v: v)):
            ref = lin2(torch.tanh(lin1(fn(x))))
            if torch.allclose(ref, y0, rtol=tol, atol=tol):
                return MlpSpec(lin1, lin2, phi, d, lin1.out_features)
    return None


def _tableau_struct(scheme):
    tab = _lib.RKTableau()
    tab.s = scheme.s
    tab.fsal = 1 if scheme.fsal else 0
    tab.has_be = 1 if scheme.bembed is not None else 0
    tab.order = scheme.order
    for i in range(scheme.s):
        tab.b[i] = scheme.b[i]
        tab.c[i] = scheme.c[i]
        tab.be[i] = scheme.bembed[i] if scheme.bembed is not None else 0.0
        for j in range(scheme.s):
            tab.a[i][j] = scheme.A[i][j]
    return tab


class FusedMlpRK:
    """Whole-sweep launches for a recognised MLP under a fixed-step explicit RK scheme."""

    def __init__(self, spec, scheme, dtype, device):
        self.lib = _lib.load()
        self.spec = spec
        self.scheme = scheme
        self.dtype = dtype
        self.device = device
        self.code = dtype_code(dtype)
        self.tab = _tableau_struct(scheme)
        self._sched_cache = {}
        self._work = None
        self.launches = 0
        # -ts_trajectory_solution_only 1: keep u_n per step ([nsteps, dim, ntraj]) instead of the s stage values; the
        # adjoint sweep recomputes the stages (pnode_mlp_rk_forward_so / _adjoint_so)
        self.solution_only = False
        # compiled hidden width the layer runs at: narrower layers are zero-padded (a padded unit adds
        # fma(0, tanh(0), acc) = acc to the slope and gets a gradient nobody reads: results are unchanged bit for bit)
        self.hidden = self.compiled_hidden(spec, scheme, dtype)
        self._pad = None
        if self.hidden != spec.hidden:
            z = dict(dtype=dtype, device=device)
            self._pad = (torch.zeros(self.hidden, spec.dim, **z), torch.zeros(self.hidden, **z),
                         torch.zeros(spec.dim, self.hidden, **z))

    COMPILED_HIDDEN = (50, 100)  # csrc/mlp_rk.cu PNODE_FOR_SHAPES

    @staticmethod
    def compiled_hidden(spec, scheme, dtype):
        lib = _lib.load()
        for h in FusedMlpRK.COMPILED_HIDDEN:
            if h >= spec.hidden and lib.pnode_mlp_rk_supported(spec.dim, h, spec.phi, dtype_code(dtype), scheme.s):
                return h
        return None

    @staticmethod
    def supported(spec, scheme, dtype):
        return FusedMlpRK.compiled_hidden(spec, scheme, dtype) is not None

    def _desc(self):
        sp = self.spec
        d = _lib.MlpDesc()
        d.dim, d.hidden, d.phi, d.dtype = sp.dim, self.hidden, sp.phi, self.code
        # live parameter storage: optimiser updates are seen by the next launch without a new setupTS
        if self._pad is None:
            d.d_w1, d.d_b1 = sp.lin1.weight.data_ptr(), sp.lin1.bias.data_ptr()
            d.d_w2 = sp.lin2.weight.data_ptr()
        else:
            w1, b1, w2 = self._pad
            h = sp.hidden
            w1[:h].copy_(sp.lin1.weight.detach())
            b1[:h].copy_(sp.lin1.bias.detach())
            w2[:, :h].copy_(sp.lin2.weight.detach())
            d.d_w1, d.d_b1, d.d_w2 = w1.data_ptr(), b1.data_ptr(), w2.data_ptr()
        d.d_b2 = sp.lin2.bias.data_ptr()
        return d

    def _unpad_mu(self, mu):
        """mu of the padded layer (W1 [hidden, dim] | b1 | W2 [dim, hidden] | b2) -> the module's parameter order and sizes."""
        if self._pad is None:
            return mu
        sp, hp = self.spec, self.hidden
        h, dm = sp.hidden, sp.dim
        o1, o2, o3 = hp * dm, hp * dm + hp, 2 * hp * dm + hp
        return torch.cat((mu[:h * dm], mu[o1:o1 + h], mu[o2:o3].view(dm, hp)[:, :h].reshape(-1), mu[o3:]))

    def _schedule(self, times, step_size):
        key = (tuple(times), tuple(step_size) if isinstance(step_size, list) else float(step_size))
        hit = self._sched_cache.get(key)
        if hit is not None:
            return hit
        loop, steps = fixed_schedule(times, step_size, self.dtype == torch.float64)
        loop.check_complete()
        arr = np.zeros(len(steps), dtype=_STEP_DTYPE)
        single = len(times) == 1
        for n, (t, h, slot) in enumerate(steps):
            arr[n]["t"], arr[n]["h"] = t, h
            if single:
                arr[n]["out_slot"] = 0 if n == len(steps) - 1 else -1
                arr[n]["in_slot"] = -1
            else:
                arr[n]["out_slot"] = slot
                arr[n]["in_slot"] = 0 if n == 0 else steps[n - 1][2]
        dev = torch.from_numpy(arr.view(np.uint8)).to(self.device)
        entry = (dev, len(steps), loop)
        if len(self._sched_cache) > 64:
            self._sched_cache.clear()
        self._sched_cache[key] = entry
        return entry

    def forward(self, u0, times, step_size, save):
        """u0: flat [ntraj*dim].  Returns (sol [T, ntraj*dim], ckpt or None, schedule entry)."""
        sp = self.spec
        ntraj = u0.numel() // sp.dim
        sched, nsteps, loop = self._schedule(times, step_size)
        T = len(times)
        sol = torch.empty((T, u0.numel()), dtype=self.dtype, device=self.device)
        if T > 1:
            sol[0].copy_(u0)
        ckpt = None
        so = bool(self.solution_only and save)
        desc = self._desc()
        if save:
            rows = int(self.lib.pnode_mlp_rk_ckpt_rows(C.byref(desc), C.byref(self.tab)))
            shape = (max(nsteps, 1), sp.dim, ntraj) if so else (max(nsteps, 1), self.scheme.s, rows, ntraj)
            ckpt = torch.empty(shape, dtype=self.dtype, device=self.device)
        if nsteps == 0:
            sol[-1].copy_(u0)
        fwd = self.lib.pnode_mlp_rk_forward_so if so else self.lib.pnode_mlp_rk_forward
        _lib.check(fwd(C.byref(desc), C.byref(self.tab), u0.data_ptr(), ntraj, sched.data_ptr(), nsteps, sol.data_ptr(),
                       None if ckpt is None else ckpt.data_ptr(), _stream()))
        self.launches += 1
        return sol, ckpt, (sched, nsteps, loop)

    def adjoint(self, gout, ckpt, sched_entry, ntraj, comm=None):
        """gout: contiguous [T, ntraj*dim].  Returns (lambda [ntraj*dim], mu [np], reduced) -- `reduced` tells the caller
        that mu is already summed over the ranks of `comm` (in-kernel peer-memory all-reduce)."""
        sp = self.spec
        sched, nsteps, _ = sched_entry
        T = gout.shape[0]
        lam = torch.empty(ntraj * sp.dim, dtype=self.dtype, device=self.device)
        npar = 2 * self.hidden * sp.dim + self.hidden + sp.dim
        mu = torch.empty(npar, dtype=self.dtype, device=self.device)
        desc = self._desc()
        if self._work is None:
            nbytes = int(self.lib.pnode_mlp_rk_adjoint_work_bytes(C.byref(desc)))
            self._work = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
        if nsteps == 0:
            lam.copy_(gout[-1])
            mu.zero_()
            return lam, self._unpad_mu(mu), False
        peer = getattr(comm, "peer", None) if comm is not None else None
        if ckpt.dim() == 3:  # solution checkpoints ([nsteps, dim, ntraj]): the sweep recomputes the stages
            _lib.check(self.lib.pnode_mlp_rk_adjoint_so(
                C.byref(desc), C.byref(self.tab), ntraj, sched.data_ptr(), nsteps, T - 1, gout.data_ptr(), ckpt.data_ptr(),
                lam.data_ptr(), mu.data_ptr(), self._work.data_ptr(), None if peer is None else peer["ptrs_dev"],
                comm.rank if peer is not None else 0, comm.world if peer is not None else 1,
                comm.next_epoch() if peer is not None else 0, _stream()))
        elif peer is not None:
            _lib.check(self.lib.pnode_mlp_rk_adjoint_dp(C.byref(desc), C.byref(self.tab), ntraj, sched.data_ptr(), nsteps,
                                                        T - 1, gout.data_ptr(), ckpt.data_ptr(), lam.data_ptr(),
                                                        mu.data_ptr(), self._work.data_ptr(), peer["ptrs_dev"], comm.rank,
                                                        comm.world, comm.next_epoch(), _stream()))
        else:
            _lib.check(self.lib.pnode_mlp_rk_adjoint(C.byref(desc), C.byref(self.tab), ntraj, sched.data_ptr(), nsteps,
                                                     T - 1, gout.data_ptr(), ckpt.data_ptr(), lam.data_ptr(),
                                                     mu.data_ptr(), self._work.data_ptr(), _stream()))
        self.launches += 1
        return lam, self._unpad_mu(mu), peer is not None


# ----------------------------------------------------------------------------------------------------------------------
# FFJORD continuous normalising flow (BASELINE config 3): csrc/cnf_rk.cu


class CnfSpec:
    """A recognised FFJORD right-hand side: ODEfunc `odefunc` over L ConcatSquashLinear `layers` (widths `dims`, dims[0] =
    dims[L] = D) and a batch of B samples.  `l1`, `l2`, `hidden` describe the two-layer shape of the fused sweeps.  `trace`
    is what the module's divergence computes: "hutchinson" (e^T J e, divergence_approx) or "exact" (tr J, divergence_bf)."""

    def __init__(self, odefunc, layers, batch, dim):
        self.odefunc, self.layers = odefunc, list(layers)
        self.batch, self.dim = batch, dim
        self.dims = [dim] + [m._layer.out_features for m in self.layers]
        self.l1, self.l2, self.hidden = self.layers[0], self.layers[-1], self.dims[1]
        self.t_via_f32 = 1
        self.trace = "hutchinson"

    @staticmethod
    def layer_params(m):
        return [m._layer.weight, m._layer.bias, m._hyper_bias.weight, m._hyper_gate.weight, m._hyper_gate.bias]

    def params(self):
        out = []
        for m in self.layers:
            out += self.layer_params(m)
        return out


# odefunc -> {(id(diffeq), dims, dtype, device, training): (weakref to diffeq, t_via_f32, trace)} once the numerical probe has
# passed.  Weak in both modules: a verdict must not pass to a new module that CPython places at the address of a freed one.
# The training flag is part of the key because FFJORD's ODEfunc switches to the exact trace in eval mode for 2-D states.
_CNF_RECOGNISED = weakref.WeakKeyDictionary()


def _is_concatsquash(m):
    return (isinstance(getattr(m, "_layer", None), nn.Linear) and isinstance(getattr(m, "_hyper_bias", None), nn.Linear)
            and isinstance(getattr(m, "_hyper_gate", None), nn.Linear) and m._hyper_bias.bias is None
            and m._hyper_gate.bias is not None and m._layer.bias is not None and m._hyper_bias.in_features == 1
            and m._hyper_gate.in_features == 1)


def cnf_closed_form(layers, z, e, t, exact=False):
    """(f, div) of the ConcatSquash network at time tensor t, the Hutchinson trace div = e^T (df/dz) e formed as the forward
    tangent of e -- the formula csrc/cnf_net.cu evaluates (and, for two layers, csrc/cnf_rk.cu).  With exact=True, div is
    the exact trace tr(df/dz), the sum of the diagonals of the forward tangents of the D unit vectors (e is not read)."""
    B, D = z.shape
    x = z
    v = torch.eye(D, dtype=z.dtype, device=z.device)[:, None, :].expand(D, B, D) if exact else e[None]
    for l, m in enumerate(layers):
        gam = torch.sigmoid(m._hyper_gate(t.view(1, 1)))
        a = m._layer(x) * gam + m._hyper_bias(t.view(1, 1))
        u = (v @ m._layer.weight.T) * gam
        if l < len(layers) - 1:
            x = torch.nn.functional.softplus(a)
            v = torch.where(a > 20, torch.ones_like(a), torch.sigmoid(a)) * u
    if exact:
        return a, torch.diagonal(u, dim1=0, dim2=2).sum(1)
    return a, (e * u[0]).sum(1)


def hutchinson_probe(bf, batch, dim, dtype, device):
    """The Hutchinson probe of ODEfunc `bf` as the kernels read it.  When absent it is drawn the way the module draws it in
    the first evaluation of a solve (odefunc.py:359-364); it is kept on the module in the state's dtype and device."""
    if getattr(bf, "_e", None) is None:
        z0 = torch.empty(batch, dim, dtype=dtype, device=device)
        bf._e = torch.randint(0, 2, z0.shape, device=device).to(z0) * 2 - 1 if getattr(bf, "rademacher", False) \
            else torch.randn_like(z0)
    e = bf._e
    if e.dtype != dtype or e.device != device or not e.is_contiguous():
        e = e.to(device=device, dtype=dtype).contiguous()
        bf._e = e
    return e


def recognise_cnf(func, u_meta):
    """Match the object graph cnf.py:72-80 builds -- FlattenFunc(base_func=ODEfunc(diffeq=ODEnet(L >= 1 ConcatSquashLinear
    layers with Softplus between them), divergence_approx or divergence_bf, residual=False), y0=(z [B,D], logp [B,1])) -- by
    duck typing, then confirm with a numerical probe that func(t, y) equals cnf_closed_form (once per diffeq module and
    training flag).  The probe, not the divergence_fn attribute, decides the trace kind: FFJORD's ODEfunc takes the exact
    trace in eval mode for 2-D states whatever its divergence_fn.  Which runner evaluates it (the two-layer fused sweeps
    for the Hutchinson trace, or the evaluator of any depth) is decided where the runner is chosen."""
    bf, y0 = getattr(func, "base_func", None), getattr(func, "y0", None)
    if bf is None or not isinstance(y0, (tuple, list)) or len(y0) != 2 or not u_meta.is_cuda:
        return None
    z0, l0 = y0
    if z0.dim() != 2 or l0.numel() != z0.shape[0] or u_meta.dim() != 1 or u_meta.numel() != z0.numel() + l0.numel():
        return None
    net = getattr(bf, "diffeq", None)
    layers = getattr(net, "layers", None)
    acts = getattr(net, "activation_fns", None)
    if layers is None or acts is None or len(layers) < 1 or len(acts) != len(layers) - 1 or \
            getattr(net, "num_squeeze", 0) != 0:
        return None
    if not all(_is_concatsquash(l) for l in layers) or not all(isinstance(a, nn.Softplus) for a in acts):
        return None
    if any(a.beta != 1 or a.threshold != 20 for a in acts) or getattr(bf, "residual", False):
        return None
    if getattr(getattr(bf, "divergence_fn", None), "__name__", "") not in ("divergence_approx", "divergence_bf"):
        return None
    B, D = z0.shape
    layers = list(layers)
    if layers[0]._layer.in_features != D or layers[-1]._layer.out_features != D or \
            any(a._layer.out_features != b._layer.in_features for a, b in zip(layers[:-1], layers[1:])):
        return None
    spec = CnfSpec(bf, layers, B, D)
    plist = [p for p in func.parameters() if p.requires_grad]
    want = spec.params()
    if len(plist) != len(want) or any(a is not b for a, b in zip(plist, want)):
        return None
    if any(p.dtype != u_meta.dtype or p.device != u_meta.device or not p.is_contiguous() for p in want):
        return None
    seen = _CNF_RECOGNISED.setdefault(bf, {})
    key = (id(net), tuple(spec.dims), u_meta.dtype, str(u_meta.device), bool(bf.training))
    if key not in seen or seen[key][0]() is not net:
        # probe through the user's module itself (FlattenFunc -> ODEfunc -> ODEnet), on a small batch, at times that are
        # not representable in float32 so that the module's handling of `t` is observable
        e_saved = getattr(bf, "_e", None)
        nevals = getattr(bf, "_num_evals", None)
        nevals = nevals.clone() if isinstance(nevals, torch.Tensor) else None
        nb = min(B, 8)
        try:
            with torch.no_grad():
                g = torch.Generator(device="cpu").manual_seed(4321)
                z = torch.randn(nb, D, generator=g, dtype=torch.float64).to(u_meta)
                e = torch.randn(nb, D, generator=g, dtype=torch.float64).to(u_meta)
                bf._e = e
                tol = 2e-4 if u_meta.dtype == torch.float32 else 1e-11
                verdict = None
                got = [type(func)(bf, (z, torch.zeros(nb, 1).to(u_meta)))(tval, torch.cat((z.reshape(-1),
                                                                           torch.zeros(nb).to(u_meta)))).detach()
                       for tval in (0.3, 0.9)]
                for trace in ("hutchinson", "exact"):
                    for via_f32 in (1, 0):
                        ok = True
                        for tval, g_t in zip((0.3, 0.9), got):
                            t = torch.tensor(tval).to(u_meta) if via_f32 else \
                                torch.tensor(tval, dtype=torch.float64).to(u_meta)
                            f, div = cnf_closed_form(layers, z, e, t, exact=trace == "exact")
                            ref = torch.cat((f.reshape(-1), -div))
                            ok = ok and g_t.shape == ref.shape and torch.allclose(g_t, ref, rtol=tol, atol=tol)
                        if ok:
                            verdict = (via_f32, trace)
                            break
                    if verdict is not None:
                        break
        except Exception:
            verdict = None
        finally:
            bf._e = e_saved
            if nevals is not None:
                bf._num_evals.copy_(nevals)  # the probe is not an evaluation of the user's solve
        if verdict is None:
            return None
        seen[key] = (weakref.ref(net),) + verdict
    spec.t_via_f32, spec.trace = seen[key][1], seen[key][2]
    return spec


class FusedCnfRK:
    """One launch per step attempt (all stages + error norm), one launch for the whole adjoint sweep."""

    def __init__(self, spec, scheme, dtype, device):
        from .controller import TimeLoop  # noqa: F401  (documented dependency)

        self.lib = _lib.load()
        self.spec, self.scheme, self.dtype, self.device = spec, scheme, dtype, device
        self.code = dtype_code(dtype)
        self.tab = _tableau_struct(scheme)
        self.s_eff = scheme.s - 1 if scheme.fsal else scheme.s
        self._wrms_work = torch.zeros(16 * 4 + 148 * 8 * 8, dtype=torch.uint8, device=device)
        self._sumsq = torch.zeros(1, dtype=torch.float64, device=device)
        self._adj_work = None
        self._ckpt = None
        self._ctl_key = None
        self.device_controller = True  # -pnode_device_controller 0 falls back to one host read per attempt
        self.launches = 0

    @staticmethod
    def supported(spec, scheme, dtype):
        """The sweeps carry the Hutchinson trace only: an exact-trace module takes the evaluator of any depth."""
        if spec.trace != "hutchinson" or len(spec.layers) != 2:
            return False
        return bool(_lib.load().pnode_cnf_rk_supported(spec.dim, spec.hidden, dtype_code(dtype), scheme.s))

    def _desc(self):
        sp = self.spec
        e = hutchinson_probe(sp.odefunc, sp.batch, sp.dim, self.dtype, self.device)
        d = _lib.CnfDesc()
        d.dim, d.hidden, d.dtype, d.t_via_f32 = sp.dim, sp.hidden, self.code, sp.t_via_f32
        names = ("d_w1", "d_b1", "d_hb1", "d_hgw1", "d_hgb1", "d_w2", "d_b2", "d_hb2", "d_hgw2", "d_hgb2")
        for n, p in zip(names, sp.params()):
            setattr(d, n, p.data_ptr())
        d.d_e = e.data_ptr()
        self._e_keepalive = e
        return d

    def _ckpt_buffer(self, nsteps_cap, ntraj):
        per_step = self.s_eff * self.spec.dim * ntraj
        need = nsteps_cap * per_step
        if self._ckpt is None or self._ckpt.numel() < need:
            new = torch.empty(need, dtype=self.dtype, device=self.device)
            if self._ckpt is not None and self._keep > 0:
                new[: self._keep * per_step].copy_(self._ckpt[: self._keep * per_step])
            self._ckpt = new
        return per_step

    def forward(self, u0, loop, atol, rtol, save, comm=None):
        """u0 flat [B*(D+1)].  `loop` is a controller.TimeLoop.  Returns (sol dict, state)."""
        if loop.adaptive and torch.cuda.is_current_stream_capturing():
            return self._forward_captured(u0, loop, atol, rtol, save, comm)
        peer = getattr(comm, "peer", None) if comm is not None else None
        sharded_ok = comm is None or peer is not None  # in-kernel all-reduce of the error norm
        if self.device_controller and loop.adaptive and sharded_ok and loop.step_list is None and \
                (loop.span is None or len(loop.span) <= _lib.CTL_MAX_SPAN) and self.scheme.bembed is not None:
            return self._forward_device_ctl(u0, loop, atol, rtol, save, comm)
        sp = self.spec
        ntraj = sp.batch
        n = u0.numel()
        n_global = n if comm is None else comm.global_count(n)
        desc = self._desc()
        u = u0.clone()
        unew = torch.empty_like(u)
        k_in, k_out = None, (torch.empty_like(u) if self.scheme.fsal else None)
        k_spare = torch.empty_like(u) if self.scheme.fsal else None
        sols = {0: u0} if loop.span is not None else {}
        steps = []
        self._keep = 0
        cap = 16
        per_step = self._ckpt_buffer(cap, ntraj) if save else 0
        esz = u.element_size()
        while not loop.done:
            t, h = loop.t, loop.h
            if save and len(steps) >= cap:
                self._keep = len(steps)
                cap *= 2
                per_step = self._ckpt_buffer(cap, ntraj)
            ck = (self._ckpt.data_ptr() + len(steps) * per_step * esz) if save else None
            _lib.check(self.lib.pnode_cnf_rk_attempt(
                C.byref(desc), C.byref(self.tab), u.data_ptr(), None if k_in is None else k_in.data_ptr(), ntraj,
                float(t), float(h), unew.data_ptr(), None if k_out is None else k_out.data_ptr(), ck, float(atol),
                float(rtol), self._sumsq.data_ptr() if loop.adaptive else None, self._wrms_work.data_ptr(), _stream()))
            self.launches += 1
            enorm = None
            if loop.adaptive:
                if comm is not None:
                    comm.allreduce_scalar(self._sumsq)
                enorm = (float(self._sumsq.item()) / n_global) ** 0.5  # the one host read per attempt
            if not loop.report(enorm):
                continue  # rejected: u and the carried-over slope k_in are unchanged
            steps.append((t, h, loop.last_out_slot))
            u, unew = unew, u
            if self.scheme.fsal:
                k_in, k_out, k_spare = k_out, k_spare, (k_in if k_in is not None else torch.empty_like(u))
            if loop.last_out_slot >= 0:
                sols[loop.last_out_slot] = u.clone()
        loop.check_complete()
        state = {"steps": steps, "ckpt": self._ckpt if save else None, "ntraj": ntraj, "desc_keep": desc,
                 "e_keep": self._e_keepalive}  # the descriptor points into this solve's probe tensor
        if save:
            self._ckpt = None  # ownership moves to the autograd node; the next solve allocates afresh
        return u, sols, state

    # ---- adaptive run with the accept/reject decision and the next step size taken ON THE DEVICE --------------------------
    CKPT_STEPS0 = 16  # checkpoint room of a fresh buffer, in steps (doubled when a solve runs out of it)

    class _Lease:
        """A checkpoint buffer and a copy of the Hutchinson probe on loan to one solve's autograd state; they go back to the
        pool when that state dies, so solves of the same shape keep presenting the same addresses to the cached loop graphs
        (csrc/cnf_rk.cu) -- FFJORD's driver draws a fresh probe tensor for every forward (cnf.py: before_odeint), and a
        backward must still see the probe of ITS forward when other solves ran in between."""

        def __init__(self, pool, buf, ebuf):
            self.pool, self.buf, self.ebuf = pool, buf, ebuf

        def __del__(self):
            pool = self.pool
            if pool is not None and len(pool) < 4:
                pool.append((self.buf, self.ebuf))

    def _ctl_buffers(self, n, nspan):
        key = (n, nspan)
        if self._ctl_key != key:
            self._ctl_key = key
            nbytes = C.sizeof(_lib.CnfCtl)
            self._ctl_host = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
            self._ctl_dev = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
            self._ctl_view = _lib.CnfCtl.from_buffer(self._ctl_host.numpy())
            self._ubuf = torch.empty(2, n, dtype=self.dtype, device=self.device)
            self._kbuf = torch.empty(2, n, dtype=self.dtype, device=self.device) if self.scheme.fsal else None
            self._solbuf = torch.empty(nspan, n, dtype=self.dtype, device=self.device) if nspan else None
            self._ckpt_pool = []
        return self._ubuf, self._kbuf, self._solbuf

    def _forward_device_ctl(self, u0, loop, atol, rtol, save, comm=None):
        """Same contract as forward().  The attempt kernel's last block runs TSAdaptChoose_Basic + MATCHSTEP + the span
        bookkeeping (csrc/cnf_rk.cu, namespace ctl) and publishes (t, h, buffers) for the next attempt.  The whole time
        loop is ONE launch -- a CUDA graph whose WHILE node repeats the attempt kernel until the controller says stop
        (pnode_cnf_rk_solve_ctl) -- and the host reads the control block once per solve; the host TimeLoop then follows
        the device's log (TimeLoop.follow) for the bookkeeping the caller reads."""
        sp = self.spec
        ntraj = sp.batch
        n = u0.numel()
        desc = self._desc()
        nspan = 0 if loop.span is None else len(loop.span)
        ubuf, kbuf, sol = self._ctl_buffers(n, nspan)
        ubuf[0].copy_(u0)
        per_step = self.s_eff * sp.dim * ntraj
        buf, ebuf = self._ckpt_pool.pop() if self._ckpt_pool else (None, None)
        if save and buf is None:
            buf = torch.empty(self.CKPT_STEPS0 * per_step, dtype=self.dtype, device=self.device)
        if ebuf is None:
            ebuf = torch.empty(ntraj * sp.dim, dtype=self.dtype, device=self.device)
        lease = self._Lease(self._ckpt_pool, buf, ebuf)
        ebuf.copy_(self._e_keepalive.reshape(-1))
        desc.d_e = ebuf.data_ptr()
        cap = buf.numel() // per_step if save else 0
        ctl = _lib.CnfCtl()
        ctl.t, ctl.h, ctl.t_end, ctl.dt_span_cached = loop.t, loop.h, loop.t_end, 0.0
        for i in range(nspan):
            ctl.span[i] = loop.span[i]
        peer = getattr(comm, "peer", None) if comm is not None else None
        ctl.n_global, ctl.delta = float(n if comm is None else comm.global_count(n)), loop.delta
        if peer is not None:
            # sharded: the ranks' loops meet in every attempt (error norm summed over NVLink inside the kernel); the
            # collective numbers continue the communicator's sequence and are handed back after the solve
            ctl.epoch_next = peer["epoch"] + 1
        ctl.nspan, ctl.order, ctl.max_reject = nspan, int(loop.order), int(loop.max_reject)
        ctl.done = 1 if loop.done else 0
        ctl.prev_ok, ctl.ctr, ctl.cur_sol_index, ctl.pending_slot = 1, 1, 1, -1
        ctl.max_steps, ctl.single, ctl.prev_out_slot = cap, 0, -1
        host_view = self._ctl_view
        nread = _lib.CnfCtl.sched.offset  # the host reads state + attempt log; the device-side schedule stays on the device
        head = _lib.CnfCtl.log_t.offset  # everything before the log is the controller's state
        stream = torch.cuda.current_stream()

        def upload(src):
            C.memmove(C.addressof(host_view), C.addressof(src), head)
            self._ctl_dev[:head].copy_(self._ctl_host[:head], non_blocking=True)

        upload(ctl)
        sols = {0: u0} if nspan else {}
        steps = []
        seen = 0
        c = host_view
        while not loop.done:
            args = (C.byref(desc), C.byref(self.tab), ubuf.data_ptr(), None if kbuf is None else kbuf.data_ptr(), ntraj,
                    lease.buf.data_ptr() if save else None, per_step, None if sol is None else sol.data_ptr(), float(atol),
                    float(rtol), self._ctl_dev.data_ptr(), self._wrms_work.data_ptr())
            if peer is not None:
                _lib.check(self.lib.pnode_cnf_rk_solve_ctl_dp(*args, peer["ptrs_dev"], comm.rank, comm.world,
                                                              stream.cuda_stream))
            else:
                _lib.check(self.lib.pnode_cnf_rk_solve_ctl(*args, stream.cuda_stream))
            self._ctl_host[:nread].copy_(self._ctl_dev[:nread], non_blocking=True)
            stream.synchronize()  # the one host read per solve
            now = c.attempts
            if peer is not None:
                comm.collectives += int(c.epoch_next) - 1 - peer["epoch"]
                peer["epoch"] = int(c.epoch_next) - 1
            self.launches += now - seen  # kernel nodes the graph's WHILE loop executed
            for a in range(seen, now):
                last = a + 1 == now
                t_next = c.t if last else c.log_t[a + 1]
                h_next = c.h if last else c.log_h[a + 1]
                t, h = loop.t, loop.h
                if loop.follow(bool(c.log_accepted[a]), c.log_enorm[a], t_next, h_next):
                    steps.append((t, h, loop.last_out_slot))
            seen = now
            if c.done == 2:
                raise RuntimeError("TS_DIVERGED_STEP_REJECTED: %d consecutive rejections at t=%g" % (c.rejections, c.t))
            if c.done in (3, 4):  # attempt log full / out of checkpoint room: make room and go on
                keep = _lib.CnfCtl()
                C.memmove(C.addressof(keep), C.addressof(c), head)
                if c.done == 3:
                    keep.attempts = 0
                    seen = 0
                else:
                    grown = torch.empty(2 * lease.buf.numel(), dtype=self.dtype, device=self.device)
                    grown[: len(steps) * per_step].copy_(lease.buf[: len(steps) * per_step])
                    lease.buf = grown  # the bigger buffer is the one that returns to the pool
                    keep.max_steps = grown.numel() // per_step
                keep.done = 0
                upload(keep)
        assert c.steps == len(steps) or not steps, "device controller and host bookkeeping disagree on the step count"
        u = ubuf[c.cur].clone() if steps else u0.clone()
        for t_h_slot in steps:
            slot = t_h_slot[2]
            if slot >= 0:
                # the state that landed on the LAST output time is the final one; earlier slots were copied by the
                # attempt that followed them
                sols[slot] = u if t_h_slot is steps[-1] else sol[slot].clone()
        loop.check_complete()
        state = {"steps": steps, "ckpt": lease.buf if save else None, "ntraj": ntraj, "desc_keep": desc, "lease": lease}
        if not save:
            state["lease"] = None  # nothing will run an adjoint on this solve: the buffers go back at once
        return u, sols, state

    CAPTURE_ATTEMPTS = 24  # -pnode_capture_attempts: attempt budget of an adaptive solve recorded into a CUDA graph

    def _forward_captured(self, u0, loop, atol, rtol, save, comm):
        """An adaptive solve while the caller records a CUDA graph (torch.cuda.graph around the training step): nothing may
        read the device, so a fixed budget of attempts is recorded (those after the end time return at once), the states at
        the output times are gathered on the device, and the adjoint sweep will take its schedule from the control block
        (pnode_cnf_rk_adjoint_ctl).  A replay whose solve needs more attempts than the budget returns NaN, not a wrong
        answer.  The host TimeLoop is not advanced: `ode._loop` statistics describe eager solves only."""
        if comm is not None or loop.step_list is not None or self.scheme.bembed is None or loop.span is None or \
                len(loop.span) > _lib.CTL_MAX_SPAN or not self.device_controller:
            raise Error(-60, "this adaptive solve cannot be recorded into a CUDA graph (needs the device step controller, "
                             "a single rank, a scalar step size and 2..%d output times)" % _lib.CTL_MAX_SPAN)
        sp = self.spec
        ntraj, n, nspan = sp.batch, u0.numel(), len(loop.span)
        nb = int(self.CAPTURE_ATTEMPTS)
        if not (1 <= nb <= _lib.CTL_MAX_LOG):
            raise Error(-60, "-pnode_capture_attempts must be in 1..%d" % _lib.CTL_MAX_LOG)
        desc = self._desc()
        per_step = self.s_eff * sp.dim * ntraj
        dev = self.device
        ubuf = torch.empty(2, n, dtype=self.dtype, device=dev)
        kbuf = torch.empty(2, n, dtype=self.dtype, device=dev) if self.scheme.fsal else None
        sol = torch.empty(nspan, n, dtype=self.dtype, device=dev)
        ckpt = torch.empty(nb * per_step, dtype=self.dtype, device=dev) if save else None
        ebuf = torch.empty(ntraj * sp.dim, dtype=self.dtype, device=dev)
        ebuf.copy_(self._e_keepalive.reshape(-1))
        desc.d_e = ebuf.data_ptr()
        ctl = _lib.CnfCtl()
        ctl.t, ctl.h, ctl.t_end, ctl.dt_span_cached = loop.t, loop.h, loop.t_end, 0.0
        for i in range(nspan):
            ctl.span[i] = loop.span[i]
        ctl.n_global, ctl.delta = float(n), loop.delta
        ctl.nspan, ctl.order, ctl.max_reject = nspan, int(loop.order), int(loop.max_reject)
        ctl.prev_ok, ctl.ctr, ctl.cur_sol_index, ctl.pending_slot = 1, 1, 1, -1
        ctl.max_steps, ctl.single, ctl.prev_out_slot = nb if save else 0, 0, -1
        head = _lib.CnfCtl.log_t.offset
        pinned = torch.empty(head, dtype=torch.uint8).pin_memory()  # re-read by the copy node at every replay
        C.memmove(pinned.data_ptr(), C.addressof(ctl), head)
        ctl_dev = torch.empty(C.sizeof(_lib.CnfCtl), dtype=torch.uint8, device=dev)
        ctl_dev[:head].copy_(pinned, non_blocking=True)
        ubuf[0].copy_(u0)
        stream = torch.cuda.current_stream().cuda_stream
        left = nb
        while left > 0:
            k = min(left, 64)
            _lib.check(self.lib.pnode_cnf_rk_attempts_ctl(
                C.byref(desc), C.byref(self.tab), ubuf.data_ptr(), None if kbuf is None else kbuf.data_ptr(), ntraj,
                None if ckpt is None else ckpt.data_ptr(), per_step, sol.data_ptr(), float(atol), float(rtol),
                ctl_dev.data_ptr(), self._wrms_work.data_ptr(), k, stream))
            left -= k
        self.launches += nb
        out = torch.empty(nspan, n, dtype=self.dtype, device=dev)
        out[0].copy_(u0)
        _lib.check(self.lib.pnode_cnf_rk_gather_ctl(ctl_dev.data_ptr(), ubuf.data_ptr(), sol.data_ptr(), out.data_ptr(), nspan, n,
                                                    self.code, stream))
        sols = {k: out[k] for k in range(nspan)}
        state = {"captured": True, "ctl": ctl_dev, "ckpt": ckpt, "ntraj": ntraj, "desc_keep": desc, "steps": [],
                 "keep": (pinned, ubuf, kbuf, sol, ebuf, out)}
        return out[nspan - 1], sols, state

    def _adjoint_captured(self, gout, state):
        sp = self.spec
        ntraj = state["ntraj"]
        npar = 2 * sp.hidden * sp.dim + 4 * sp.hidden + 4 * sp.dim
        lam = torch.empty(ntraj * (sp.dim + 1), dtype=self.dtype, device=self.device)
        mu = torch.empty(npar, dtype=self.dtype, device=self.device)
        desc = state["desc_keep"]
        if "adj_work" not in state:  # owned by the recorded solve (allocated from the graph's pool when recording)
            state["adj_work"] = torch.zeros(int(self.lib.pnode_cnf_rk_adjoint_work_bytes(C.byref(desc))), dtype=torch.uint8,
                                            device=self.device)
        _lib.check(self.lib.pnode_cnf_rk_adjoint_ctl(C.byref(desc), C.byref(self.tab), ntraj, state["ctl"].data_ptr(),
                                                     gout.shape[0] - 1, gout.data_ptr(), state["ckpt"].data_ptr(),
                                                     lam.data_ptr(), mu.data_ptr(), state["adj_work"].data_ptr(), _stream()))
        self.launches += 1
        return lam, mu, False

    def adjoint(self, gout, state, single, nadj=None, comm=None):
        """gout contiguous [T, B*(D+1)].  `nadj`: run only the last nadj steps (the reference's one-element-t rule).
        Returns (lambda, mu, reduced)."""
        if state.get("captured"):
            return self._adjoint_captured(gout, state)
        sp = self.spec
        steps, ntraj = state["steps"], state["ntraj"]
        first = 0 if nadj is None else max(len(steps) - nadj, 0)
        steps = steps[first:]
        nsteps = len(steps)
        T = gout.shape[0]
        npar = 2 * sp.hidden * sp.dim + 4 * sp.hidden + 4 * sp.dim
        lam = torch.empty(ntraj * (sp.dim + 1), dtype=self.dtype, device=self.device)
        mu = torch.empty(npar, dtype=self.dtype, device=self.device)
        if nsteps == 0:
            lam.copy_(gout[-1])
            mu.zero_()
            return lam, mu, False
        arr = np.zeros(nsteps, dtype=_STEP_DTYPE)
        for i, (t, h, slot) in enumerate(steps):
            arr[i]["t"], arr[i]["h"] = t, h
            arr[i]["out_slot"] = slot
            arr[i]["in_slot"] = -1 if single else (0 if i == 0 else steps[i - 1][2])
        sched = torch.from_numpy(arr.view(np.uint8)).to(self.device)
        desc = state.get("desc_keep") or self._desc()  # the forward's descriptor: same weights, same probe
        per_step_bytes = self.s_eff * sp.dim * ntraj * gout.element_size()
        if self._adj_work is None:
            self._adj_work = torch.zeros(int(self.lib.pnode_cnf_rk_adjoint_work_bytes(C.byref(desc))), dtype=torch.uint8,
                                         device=self.device)
        peer = getattr(comm, "peer", None) if comm is not None else None
        args = (C.byref(desc), C.byref(self.tab), ntraj, sched.data_ptr(), nsteps, T - 1, gout.data_ptr(),
                state["ckpt"].data_ptr() + first * per_step_bytes, lam.data_ptr(), mu.data_ptr(), self._adj_work.data_ptr())
        if peer is not None:
            _lib.check(self.lib.pnode_cnf_rk_adjoint_dp(*args, peer["ptrs_dev"], comm.rank, comm.world, comm.next_epoch(),
                                                        _stream()))
        else:
            _lib.check(self.lib.pnode_cnf_rk_adjoint(*args, _stream()))
        self.launches += 1
        return lam, mu, peer is not None
