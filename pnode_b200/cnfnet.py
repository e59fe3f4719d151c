"""FFJORD right-hand sides of any depth on the tensor cores: an evaluator plugged into the generic stage loop.

  * CnfNetCallbacks -- F(t, y) of FlattenFunc(ODEfunc(ODEnet)) with L ConcatSquashLinear layers, Softplus between them and
                       the Hutchinson trace (divergence_approx) or the exact trace (divergence_bf)
                       (ffjord-pnode/lib/layers/odefunc.py:21-57,345-385, cnf.py:72-80): one C call per evaluation and one
                       per adjoint stage into csrc/cnf_net.cu.  The trace is the forward tangent of the probe (or of the D
                       unit vectors, for the exact trace), so neither the forward nor the adjoint needs autograd (the
                       reference differentiates the autograd trace a second time in every adjoint stage,
                       petsc_adjoint.py:52-82,341-363; its exact trace takes D autograd calls per evaluation).  Weight gradients
                       are accumulated straight into mu; the forward keeps an activation set per stage evaluation so the
                       adjoint does not re-evaluate.
The module is recognised by fused.recognise_cnf (structure + numerical probe through the user's module)."""
import ctypes as C

import torch

from . import _lib
from .device import _stream, dtype_code
from .engine import Callbacks
from .errors import Error
from .fused import hutchinson_probe


def _desc_for(spec, dtype):
    d = _lib.CnfNetDesc()
    d.nlayers, d.dtype, d.batch, d.t_f32 = len(spec.layers), dtype_code(dtype), spec.batch, spec.t_via_f32
    d.trace = 1 if spec.trace == "exact" else 0
    for l, n in enumerate(spec.dims):
        d.dims[l] = n
    return d


class CnfNetCallbacks(Callbacks):
    @staticmethod
    def supported(spec, dtype):
        """Depth and every reduction length (widths and (1 + chains) x batch: 2B for the Hutchinson trace, (D + 1) B for
        the exact one) within what one sliced product takes."""
        if len(spec.layers) > _lib.DMLP_MAX_LAYERS:
            return False
        d = _desc_for(spec, dtype)
        return int(_lib.load().pnode_cnfnet_weight_bytes(C.byref(d))) >= 0

    def __init__(self, func, tensor_size, spec):
        super().__init__(func, tensor_size)
        self.lib = _lib.load()
        self.spec = spec
        p0 = spec.layers[0]._layer.weight
        self.dtype, self.device = p0.dtype, p0.device
        self.code = dtype_code(self.dtype)
        offs, off = {}, 0
        for p in self.params:  # mu layout = func.parameters() filtered by requires_grad (petsc_adjoint.py:603-614)
            offs[id(p)] = off
            off += p.numel()
        d = _desc_for(spec, self.dtype)
        for l, m in enumerate(spec.layers):
            for name, p in zip(("mu_w_off", "mu_b_off", "mu_hbw_off", "mu_hgw_off", "mu_hgb_off"), spec.layer_params(m)):
                getattr(d, name)[l] = offs.get(id(p), -1)
        self._desc = d
        self._refresh_pointers()
        nb = [int(self.lib.pnode_cnfnet_weight_bytes(C.byref(d))), int(self.lib.pnode_cnfnet_act_bytes(C.byref(d))),
              int(self.lib.pnode_cnfnet_work_bytes(C.byref(d)))]
        if min(nb) < 0:
            raise Error(-50, self.lib.pnode_last_error().decode())
        self._wbuf = torch.empty(nb[0], dtype=torch.uint8, device=self.device)
        self._act_bytes = nb[1]
        self._act0 = torch.empty(nb[1], dtype=torch.uint8, device=self.device)  # evaluations that are not kept
        self._work = torch.empty(nb[2], dtype=torch.uint8, device=self.device)
        self._prepared_for = None
        self._saved, self._saved_bytes, self._saved_mark = {}, 0, set()
        from .options import Options

        self._save_budget = int(float(Options().getString("pnode_cnf_save_mb", "16384")) * (1 << 20))
        self._keep = True
        self.reused_activations = 0
        self.launches = 0

    def _refresh_pointers(self):
        """Parameters are borrowed: addresses re-read at the start of every solve."""
        for l, m in enumerate(self.spec.layers):
            for name, p in zip(("d_weight", "d_bias", "d_hyper_bias", "d_gate_weight", "d_gate_bias"),
                               self.spec.layer_params(m)):
                getattr(self._desc, name)[l] = p.data_ptr()

    def _prepare(self):
        ver = tuple((p.data_ptr(), p._version) for p in self.spec.params())
        if ver != self._prepared_for:
            self._refresh_pointers()
            _lib.check(self.lib.pnode_cnfnet_prepare(C.byref(self._desc), self._wbuf.data_ptr(), _stream()))
            self._prepared_for = ver
            self.launches += len(self.spec.layers)

    def _probe(self):
        """FFJORD draws a fresh probe per solve (before_odeint): the descriptor follows the module's current one.  The
        module draws it before it picks a divergence, so it is drawn for the exact trace too (which does not read it): the
        caller's RNG stream and `_e` end up as the module leaves them."""
        sp = self.spec
        e = hutchinson_probe(sp.odefunc, sp.batch, sp.dim, self.dtype, self.device)
        self._desc.d_e = e.data_ptr()

    def _count(self):
        """ODEfunc._num_evals (read by FFJORD's NFE counters) advances once per evaluation of the module, on the device."""
        n = getattr(self.spec.odefunc, "_num_evals", None)
        if isinstance(n, torch.Tensor):
            n.add_(1)

    def begin(self, forward, keep=True, comm=None):
        super().begin(forward, keep=keep, comm=comm)
        if forward:
            self._prepared_for = None  # weights are re-sliced once per solve (an optimiser step may have changed them)
            self._saved.clear()
            self._saved_bytes = 0
            self._keep = bool(keep)
        self._prepare()

    def release(self):
        super().release()
        self._saved.clear()
        self._saved_bytes = 0

    def mark(self):
        super().mark()
        self._saved_mark = set(self._saved.keys())

    def rollback(self):
        super().rollback()
        for k in [k for k in self._saved if k not in self._saved_mark]:
            del self._saved[k]
            self._saved_bytes -= self._act_bytes

    def _forward(self, t, u, act):
        self._probe()
        out = torch.empty_like(u)
        _lib.check(self.lib.pnode_cnfnet_forward(C.byref(self._desc), self._wbuf.data_ptr(), float(t), u.data_ptr(),
                                                 out.data_ptr(), None if act is None else act.data_ptr(),
                                                 self._work.data_ptr(), _stream()))
        self.launches += 2 + len(self.spec.layers) * (3 if act is not None else 2)
        return out

    def f(self, t, u, keep=False):
        self.nfe += 1
        self._count()
        self._prepare()
        if not u.is_contiguous():
            u = u.contiguous()
        act = None
        if keep and self._keep and self._saved_bytes + self._act_bytes <= self._save_budget:
            act = torch.empty(self._act_bytes, dtype=torch.uint8, device=u.device)
            self._saved[u.data_ptr()] = (u, u._version, float(t), act)  # holding u keeps its address unique
            self._saved_bytes += self._act_bytes
        return self._forward(t, u, act)

    def _vjp(self, t, u, w, vu, mu, coef):
        self._prepare()
        ent = self._saved.get(u.data_ptr())
        if ent is not None and ent[1] == u._version and ent[2] == float(t) and ent[0].numel() == u.numel():
            act = ent[3]
            self.reused_activations += 1
            self._probe()
        else:  # no kept activation set for this point: re-evaluate like the reference does
            self._count()
            act = self._act0
            self._forward(t, u if u.is_contiguous() else u.contiguous(), act)
        if not w.is_contiguous():
            w = w.contiguous()
        _lib.check(self.lib.pnode_cnfnet_vjp(C.byref(self._desc), self._wbuf.data_ptr(), float(t), act.data_ptr(),
                                             w.data_ptr(), None if vu is None else vu.data_ptr(),
                                             None if mu is None else mu.data_ptr(), float(coef), self._work.data_ptr(),
                                             _stream()))
        self.launches += 6 * len(self.spec.layers)

    def vjp(self, t, u, w, want_u=True, want_params=True):
        self.nvjp += 1
        vu = torch.empty_like(u) if want_u else None
        mu = torch.zeros(self.nparams, dtype=u.dtype, device=u.device) if want_params and self.nparams else None
        self._vjp(t, u, w, vu, mu, 1.0)
        return vu, (list(torch.split(mu, self.sizes)) if mu is not None else [])

    def vjp_accumulate(self, t, u, w, mu, coef):
        """J^T w, and mu += coef * (df/dp)^T w inside the products' epilogues and the bias / gate finalize kernel."""
        self.nvjp += 1
        vu = torch.empty_like(u)
        if mu is not None and mu.numel() != self.nparams:
            raise Error(-51, "cnf net: mu slice has %d entries, the function has %d parameters" % (mu.numel(), self.nparams))
        self._vjp(t, u, w, vu, mu if self.nparams else None, coef)
        return vu, None
