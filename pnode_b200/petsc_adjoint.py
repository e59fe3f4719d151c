"""Drop-in mirror of the reference's `pnode/petsc_adjoint.py` public surface (class ODEPetsc: setupTS / odeint /
odeint_adjoint, reference lines 366-900; autograd bridge OdeintAdjointMethod, 903-947) on top of the B200-native engine.

Same argument names, order and defaults as petsc_adjoint.py:534-550; same behavioural contract (SURVEY.md appendix C):
  * unknown `method` strings silently keep the TS default (RK 3bs); `fixed_*` names are aliases (641-656);
  * the scheme is (re)applied only when the state's shape / dtype / device changes (627-656), while step size,
    trajectory on/off and the `-ts_*` command-line options are re-read on every call (768-775);
  * `t` with one element integrates [0, t0] and returns [1, *shape]; longer `t` returns every point (818-865);
  * `step_size` may be a per-step list (523-525, 816-817);
  * gradients: lambda <- grad[-1], forcing added after each output interval's adjoint, mu delivered to each
    parameter's .grad in `func.parameters()` order, implicit block first for IMEX (603-614, 916-947).
What differs, deliberately: tensors must live on a CUDA device (no CPU path, no DLPack/numpy staging -- `use_dlpack` is
accepted and ignored); `fixed_jacobian_across_solves` (passed by examples-sinode/KS/KS.py:494 although the reference
signature lacks it) is accepted as an alias of `fixed_jacobian`; a fused sweep never calls `func`, so `func.nfe`
counters do not advance on that path.
"""
import torch
import torch.nn as nn

from . import tableaux
from .cnfnet import CnfNetCallbacks
from .controller import TimeLoop
from .device import DeviceOps
from .convblock import ConvBlockCallbacks, recognise_convblock
from .densemlp import (CirculantCallbacks, CirculantSolver, DenseMlpCallbacks, recognise_circulant,
                       recognise_relu_mlp)
from .engine import Callbacks, GenericTS, ImplicitSolver
from .errors import Error
from .fused import FusedCnfRK, FusedMlpRK, recognise_cnf, recognise_mlp
from .options import Options


def single_time_adjoint_steps(loop):
    """petsc_adjoint.py:873-875: for a one-element `t` the reference runs round(|t / ts.getTimeStep()|) adjoint steps,
    where getTimeStep() is the step PETSc proposed AFTER the last step.  Exact for fixed steps that divide t; for adaptive
    runs it is the reference's (questionable) behaviour, reproduced here and capped by the steps actually taken."""
    h = loop.h
    n = int(round(abs(loop.t_end / h))) if h != 0 else 0
    return min(n, loop.steps)


def _on_device(device):
    """Kernels are launched on the raw stream of the CURRENT device: make the state's device current for the call."""
    import contextlib
    if device is not None and device.type == "cuda":
        return torch.cuda.device(device)
    return contextlib.nullcontext()


def _check_device(tensor, what):
    """The single gate of the product path: CUDA tensors only."""
    if not tensor.is_cuda:
        raise Error(-11, "%s must be a CUDA tensor (got device %s); pnode_b200 has no CPU fallback" %
                    (what, tensor.device))
    cur = torch.cuda.current_device()
    if tensor.device.index is not None and tensor.device.index != cur:
        # the kernels launch on the CURRENT device's current stream (device._stream): a tensor of another GPU would be read
        # unordered with respect to the torch ops that produced it, or not at all without peer access
        raise Error(-11, "%s lives on cuda:%d but the current CUDA device is cuda:%d; call torch.cuda.set_device(%d) (one "
                         "process per GPU) before using ODEPetsc" % (what, tensor.device.index, cur, tensor.device.index))


class ODEPetsc(object):
    comm = None  # reference: PETSc.COMM_SELF (petsc_adjoint.py:367).  Set to a pnode_b200.parallel.BatchComm for DP.

    def _modules_of(self, f):
        """list(f.modules()), kept per function object: FFJORD and the CIFAR driver call setupTS on every forward and the
        recursive walk was a tenth of a small-batch pass.  The walk is redone when the number of direct children changes."""
        cache = self.__dict__.setdefault("_mod_cache", {})
        ent = cache.get(id(f))
        if ent is None or ent[0]() is not f or ent[1] != len(f._modules):
            import weakref

            ent = (weakref.ref(f), len(f._modules), list(f.modules()))
            cache[id(f)] = ent
        return ent[2]

    def __init__(self):
        self.n = 0
        self.tensor_size = None
        self.tensor_dtype = None
        self.device = None
        self.mass = None
        self.funcIM = None
        self.funcEX = None
        self.npIM = None
        self.npEX = None
        self.np = None
        self.imex = None
        self.use_dlpack = True
        self.use_cuda = False
        self.linear_solver = None
        self.matrixfree_jacobian = True
        self.step_size = None
        self.enable_adjoint = True
        self._kind, self._scheme_name = tableaux.TS_DEFAULT
        self._ops = None
        self._engine = None
        self._fused = None
        self._fused_spec = None
        self._convblock_cache = {}
        self._rhs_kind = "torch"
        self._fused_kind = None
        self._fused_checked_for = None
        self._cb_ex = self._cb_im = self._imp = None
        self._loop = None
        self.path = None  # "fused-mlp-rk" | "fused-cnf-rk" | "generic[+<evaluator>-rhs]": which engine ran the last odeint

    # ------------------------------------------------------------------------------------------------------------
    def setupTS(self, u_tensor, func, step_size=0.01, enable_adjoint=True, implicit_form=False, use_dlpack=True,
                method="dopri5", mass=None, imex_form=False, func2=None, batch_size=1, linear_solver="petsc",
                fixed_jacobian=False, matrixfree_jacobian=True, fixed_jacobian_across_solves=None):
        if imex_form and func2 is None:
            raise ValueError("func2 must be provided to enable imex_form=True")
        _check_device(u_tensor, "ODEPetsc.setupTS: the state tensor")
        if fixed_jacobian_across_solves is not None:
            fixed_jacobian = bool(fixed_jacobian_across_solves)
        self.imex = imex_form
        self.linear_solver = linear_solver
        self.fixed_jacobian = fixed_jacobian
        if linear_solver == "petsc":
            matrixfree_jacobian = True
        if fixed_jacobian or linear_solver == "torch":
            matrixfree_jacobian = False
        self.matrixfree_jacobian = matrixfree_jacobian
        func_ex = func2 if imex_form else func
        funcs_changed = self.funcIM is not func or self.funcEX is not func_ex
        meta_changed = (u_tensor.size() != self.tensor_size or u_tensor.dtype != self.tensor_dtype
                        or u_tensor.device != self.device)
        # train()/eval() switches change what the modules compute (BatchNorm statistics, Dropout): the evaluators chosen below
        # -- and Callbacks' decision to keep stage graphs -- are re-derived whenever any sub-module's mode flips
        mode_sig = tuple(m.training for f in (func, func_ex) if isinstance(f, nn.Module) for m in self._modules_of(f))
        mode_changed = mode_sig != getattr(self, "_mode_sig", None)
        self._mode_sig = mode_sig
        if funcs_changed:
            self.funcIM, self.funcEX = func, func_ex
        if meta_changed:
            self.tensor_size = u_tensor.size()
            self.tensor_dtype = u_tensor.dtype
            self.device = u_tensor.device
            self.use_cuda = True
            self.n = u_tensor.numel()
            self._kind, self._scheme_name = tableaux.METHODS.get(method, tableaux.TS_DEFAULT)
            self.implicit_form = implicit_form
            self._ops = DeviceOps(self.device, self.tensor_dtype)
        if funcs_changed or meta_changed or mode_changed:
            self._cb_im = Callbacks(self.funcIM, self.tensor_size)
            self._rhs_kind = "torch"
            if not imex_form and Options().getString("pnode_fused", "1") not in ("0", "false", "no"):
                # convolutional ODE block: same generic stage loop, hand-written BN+ReLU kernels inside f / vjp
                key = (id(func), tuple(u_tensor.shape), u_tensor.dtype, mode_sig)
                if key in self._convblock_cache or recognise_convblock(func, u_tensor):
                    self._convblock_cache[key] = True
                    self._cb_im = ConvBlockCallbacks(func, self.tensor_size)
                    self._rhs_kind = "convblock"
            self._cb_ex = self._cb_im if self.funcEX is self.funcIM else Callbacks(self.funcEX, self.tensor_size)
            if Options().getString("pnode_fused", "1") not in ("0", "false", "no") and self._rhs_kind == "torch":
                # wide ReLU MLP (SINODE explicit half / plain MLP right-hand side): tensor-core evaluator
                spec = recognise_relu_mlp(self.funcEX, u_tensor)
                if spec is not None:
                    cb = DenseMlpCallbacks(self.funcEX, self.tensor_size, spec[0], spec[1])
                    if self._cb_ex is self._cb_im:
                        self._cb_im = cb
                    self._cb_ex = cb
                    self._rhs_kind = "dense-mlp"
                if spec is None and not imex_form:
                    # FFJORD network of any depth: tensor-core evaluator with the trace and its adjoint in closed form (the
                    # two-layer shapes of the fused sweeps still take those where _fused_runner picks them)
                    cnf = recognise_cnf(self.funcEX, u_tensor)
                    if cnf is not None and CnfNetCallbacks.supported(cnf, u_tensor.dtype):
                        self._cb_ex = self._cb_im = CnfNetCallbacks(self.funcEX, self.tensor_size, cnf)
                        self._rhs_kind = "cnf-net"
                if imex_form:
                    col = recognise_circulant(self.funcIM, u_tensor)
                    if col is not None:
                        self._cb_im = CirculantCallbacks(self.funcIM, self.tensor_size, col, u_tensor.dtype, u_tensor.device)
                        self._rhs_kind = (self._rhs_kind + "+circulant") if self._rhs_kind != "torch" else "circulant"
            if imex_form:
                self.npIM, self.npEX = self._cb_im.nparams, self._cb_ex.nparams
                self.np = self.npIM + self.npEX
            else:
                self.np = self.npIM = self.npEX = self._cb_ex.nparams
            self._fused_checked_for = None
        if mass is not None:
            mass = mass.to(device=u_tensor.device, dtype=u_tensor.dtype).reshape(u_tensor.numel(), u_tensor.numel())
        self.mass = mass
        self.batch_size = batch_size
        self.step_size = step_size
        self.enable_adjoint = enable_adjoint
        self._set_from_options()

    def _set_from_options(self):
        """ts.setFromOptions() (petsc_adjoint.py:775): command-line -ts_* options beat the method= argument."""
        opt = Options()
        kind, name = self._kind, self._scheme_name
        ts_type = opt.getString("ts_type")
        if ts_type is not None:
            if ts_type == "euler":
                kind, name = "rk", "1fe"
            elif ts_type == "rk":
                if kind != "rk":
                    kind, name = "rk", tableaux.RK_DEFAULT
            elif ts_type == "arkimex":
                if kind != "arkimex":
                    kind, name = "arkimex", tableaux.ARKIMEX_DEFAULT
            elif ts_type in ("cn", "beuler"):
                kind, name = ts_type, None
            else:
                raise Error(-13, "unsupported -ts_type %s" % ts_type)
        if kind == "rk" and opt.hasName("ts_rk_type"):
            name = opt.getString("ts_rk_type")
        if kind == "arkimex" and opt.hasName("ts_arkimex_type"):
            name = opt.getString("ts_arkimex_type")
        try:
            self._scheme = tableaux.lookup(kind, name)
        except KeyError as e:
            raise Error(-14, str(e))
        self._active_kind = kind
        self._atol = opt.getReal("ts_atol", 1e-4)
        self._rtol = opt.getReal("ts_rtol", 1e-4)
        self._max_reject = opt.getInt("ts_max_reject", 10)
        self._adapt_none = opt.getString("ts_adapt_type", "basic") == "none"
        self._ksponly = opt.getString("snes_type") == "ksponly"
        self._monitor = opt.hasName("ts_monitor")
        self._allow_fused = opt.getString("pnode_fused", "1") not in ("0", "false", "no")
        solver_cls = ImplicitSolver
        if isinstance(self._cb_im, CirculantCallbacks) and self.linear_solver == "torch" and self.mass is None:
            solver_cls = CirculantSolver
        self._imp = solver_cls(self._ops, self._cb_im, self.linear_solver, self.batch_size, self._ksponly,
                                   rtol=opt.getReal("snes_rtol", 1e-8), max_it=opt.getInt("snes_max_it", 50),
                                   ksp_rtol=opt.getReal("ksp_rtol", 1e-5), ksp_max_it=opt.getInt("ksp_max_it", 10000))
        self._imp.fixed_jacobian = bool(self.fixed_jacobian)
        if not hasattr(self, "_imp_cache"):
            self._imp_cache = {}
        self._imp.cache = self._imp_cache
        sol_only = opt.getString("ts_trajectory_solution_only", "0") not in ("0", "false", "no")
        max_cps = opt.getInt("ts_trajectory_max_cps_ram", None)
        if self.mass is not None and kind not in ("cn", "beuler"):
            raise Error(-12, "mass= (M u' = f) is supported for the implicit theta methods cn / beuler only, as in the "
                             "reference's DAE example (examples-pnode/pendulum_DAE.py)")
        self._imp.mass = self.mass
        self._engine = GenericTS(self._ops, self._scheme, kind, self._atol, self._rtol, comm=self.comm,
                                 solution_only=sol_only, max_cps=max_cps)
        # the fused tiny-MLP sweeps honour -ts_trajectory_solution_only themselves (u_n per step in HBM, stages recomputed
        # inside the adjoint kernel); a checkpoint budget (-ts_trajectory_max_cps_ram) and the FFJORD sweeps take the
        # generic path with those options
        self._fused_sol_only = sol_only and max_cps is None
        if max_cps is not None:
            self._allow_fused = False

    def _active_callbacks(self):
        """(explicit, implicit) right-hand sides the active scheme integrates.  Without imex_form the reference registers ONE
        function: as the IFunction when implicit_form=True, else as the RHSFunction (petsc_adjoint.py:666-730) -- an ARKIMEX
        scheme then sees an empty other half (treating the single function as both halves would integrate u' = 2 f)."""
        cb_ex, cb_im = self._cb_ex, self._cb_im
        if self._active_kind == "arkimex" and not self.imex:
            if getattr(self, "implicit_form", False):
                cb_ex = None
            else:
                cb_im = None
        return cb_ex, cb_im

    def _adaptive(self):
        if self._adapt_none or self._active_kind in ("cn", "beuler"):
            return False
        return self._scheme.bembed is not None

    def _fused_runner(self):
        """Pick a fused sweep when func is recognised: tiny-state MLP (fixed-step explicit RK) or FFJORD CNF (explicit RK,
        fixed or adaptive).  Returns (kind, runner) or None."""
        if not self._allow_fused or self._active_kind != "rk":
            return None
        key = (id(self.funcEX), self.tensor_size, self.tensor_dtype, self.device)
        if self._fused_checked_for != key:
            self._fused_checked_for = key
            meta = torch.empty(self.tensor_size, dtype=self.tensor_dtype, device=self.device)
            self._fused_spec = recognise_mlp(self.funcEX, meta)
            self._fused_kind = "mlp"
            if self._fused_spec is None:
                self._fused_spec = recognise_cnf(self.funcEX, meta)
                self._fused_kind = "cnf"
            self._fused = None
        if self._fused_spec is None:
            return None
        if self._fused_kind == "mlp":
            if self._adaptive() or not FusedMlpRK.supported(self._fused_spec, self._scheme, self.tensor_dtype):
                return None
            if self._fused is None or self._fused.scheme is not self._scheme:
                self._fused = FusedMlpRK(self._fused_spec, self._scheme, self.tensor_dtype, self.device)
            self._fused.solution_only = self._fused_sol_only
        else:
            if self._fused_sol_only:
                return None
            if not FusedCnfRK.supported(self._fused_spec, self._scheme, self.tensor_dtype):
                return None
            if self._fused is None or self._fused.scheme is not self._scheme:
                self._fused = FusedCnfRK(self._fused_spec, self._scheme, self.tensor_dtype, self.device)
            self._fused.device_controller = Options().getString("pnode_device_controller", "1") not in ("0", "false", "no")
            self._fused.CAPTURE_ATTEMPTS = Options().getInt("pnode_capture_attempts", type(self._fused).CAPTURE_ATTEMPTS)
        return self._fused_kind, self._fused

    # ------------------------------------------------------------------------------------------------------------
    def _times(self, t):
        """Output times on the host (petsc_adjoint.py:811 `t.cpu()`).  A device->host read costs a stream sync, so the list is
        kept while the caller hands in the SAME tensor object, unmodified (identity + version counter: holding the object keeps
        its address from being recycled)."""
        c = getattr(self, "_times_cache", None)
        if c is not None and c[0] is t and c[1] == t._version:
            return list(c[2])
        times = [float(x) for x in t.detach().cpu().to(dtype=torch.float64).reshape(-1)]
        self._times_cache = (t, t._version, tuple(times))
        return times

    def _odeint_impl(self, u0, t):
        with _on_device(self.device):
            return self._odeint_body(u0, t)

    def _odeint_body(self, u0, t):
        if self.tensor_size is None:
            raise Error(-15, "setupTS must be called before odeint")
        _check_device(u0, "ODEPetsc.odeint: u0")
        if u0.numel() != self.n or u0.dtype != self.tensor_dtype:
            raise Error(-16, "u0 does not match the tensor given to setupTS (numel %d vs %d, dtype %s vs %s)" %
                        (u0.numel(), self.n, u0.dtype, self.tensor_dtype))
        times = self._times(t)
        u_flat = u0.detach().reshape(-1)
        if not u_flat.is_contiguous():
            u_flat = u_flat.contiguous()
        T = len(times)
        sel = self._fused_runner()
        if sel is not None and sel[0] == "mlp":
            fused = sel[1]
            self.path = "fused-mlp-rk"
            sol, ckpt, sched = fused.forward(u_flat, times, self.step_size, self.enable_adjoint)
            self._loop = sched[2]
            state = ("fused", fused, ckpt, sched)
            return sol.view((T,) + tuple(self.tensor_size)), state
        if sel is not None and sel[0] == "cnf":
            fused = sel[1]
            self.path = "fused-cnf-rk"
            loop = TimeLoop(times, self.step_size, self._adaptive(), self._scheme.order,
                            self.tensor_dtype == torch.float64, self._max_reject)
            uf, sols, st = fused.forward(u_flat, loop, self._atol, self._rtol, self.enable_adjoint, comm=self.comm)
            self._loop = loop
            if T == 1:
                out = uf.view((1,) + tuple(self.tensor_size))
            else:
                out = torch.stack([sols[k].view(self.tensor_size) for k in range(T)], dim=0)
            st["loop"] = loop
            return out, ("fused-cnf", fused, st, T == 1)
        self.path = "generic" if self._rhs_kind == "torch" else "generic+" + self._rhs_kind + "-rhs"
        self._imp.reset()
        loop = TimeLoop(times, self.step_size, self._adaptive(), self._scheme.order if self._scheme else 1,
                        self.tensor_dtype == torch.float64, self._max_reject)
        cb_ex, cb_im = self._active_callbacks()
        if hasattr(self._cb_ex, "layer_slices"):  # sharded runs all-reduce the wide MLP's gradient layer by layer
            self._cb_ex.record_layer_events = self.comm is not None and getattr(self.comm, "world", 1) > 1
        uf, sols = self._engine.solve(cb_ex, cb_im, self._imp, u_flat, loop, self.enable_adjoint)
        self._loop = loop
        if self._monitor:
            for k, (tt, hh, ok, en) in enumerate(loop.attempts):
                print("%d TS dt %g time %g%s" % (k, hh, tt, "" if ok else " (rejected, wlte %g)" % en))
        if T == 1:
            out = uf.view((1,) + tuple(self.tensor_size))
        else:
            out = torch.stack([sols[k].view(self.tensor_size) for k in range(T)], dim=0)
        state = ("generic", loop, self._engine.traj)
        return out, state

    def odeint(self, u0, t):
        """Solves du/dt = func(t, u), u(t[0]) = u0; returns the solution at every time of `t`
        (petsc_adjoint.py:777-869)."""
        out, _ = self._odeint_impl(u0, t)
        return out

    def odeint_adjoint(self, y0, t):
        if not isinstance(self.funcIM, nn.Module):
            raise ValueError("func is required to be an instance of nn.Module.")
        params = list(self._cb_im.params)
        if self._cb_ex is not self._cb_im:
            params += list(self._cb_ex.params)
        return _OdeintAdjoint.apply(y0, t, self, *params)

    # -- TSAdjointSolve segments (petsc_adjoint.py:871-890) ----------------------------------------------------------
    def _adjoint_generic(self, loop, traj, grad, T):
        self._engine.traj = traj
        lam = grad[-1].reshape(-1).clone()
        mu = torch.zeros(self.np, dtype=self.tensor_dtype, device=self.device)
        cb_ex, cb_im = self._active_callbacks()
        np_im = self.npIM if self.imex else (self.np if cb_ex is None else 0)
        eng = self._engine
        if T == 1:
            nsteps = single_time_adjoint_steps(loop)
            nsteps = min(nsteps, len(eng.traj))
            lam = eng.adjoint_steps(cb_ex, cb_im, self._imp, nsteps, lam, mu, np_im)
        for i in range(T - 1, 0, -1):
            lam = eng.adjoint_steps(cb_ex, cb_im, self._imp, loop.cur_sol_steps[i], lam, mu, np_im)
            self._ops.lincomb(lam, lam, 1.0, [grad[i - 1].reshape(-1)], [1.0])  # forcing (petsc_adjoint.py:938)
        if not eng.traj:  # the whole trajectory has been consumed: drop what the forward kept for this sweep
            for cb in (self._cb_ex, self._cb_im):
                if cb is not None and hasattr(cb, "release"):
                    cb.release()
        return lam, mu


class _OdeintAdjoint(torch.autograd.Function):
    """OdeintAdjointMethod (petsc_adjoint.py:903-947).  The parameters are direct inputs of the Function, so mu reaches
    every Parameter.grad without the reference's flat_params cat() node."""

    @staticmethod
    def forward(ctx, y0, t, ode, *params):
        with torch.no_grad():
            ans, state = ode._odeint_impl(y0, t)
        ctx.ode = ode
        ctx.state = state
        ctx.nparams = len(params)
        ctx.shape = y0.shape
        ctx.T = ans.shape[0]
        return ans

    @staticmethod
    def backward(ctx, grad_output):
        ode = ctx.ode
        if not ode.enable_adjoint:
            raise Error(-17, "backward through odeint_adjoint needs setupTS(enable_adjoint=True)")
        T = ctx.T
        with torch.no_grad(), _on_device(ode.device):
            grad = grad_output if grad_output.is_contiguous() else grad_output.contiguous()
            if ctx.state[0] == "fused":
                _, fused, ckpt, sched = ctx.state
                ntraj = ode.n // fused.spec.dim
                lam, mu, reduced = fused.adjoint(grad.view(T, -1), ckpt, sched, ntraj, comm=ode.comm)
            elif ctx.state[0] == "fused-cnf":
                _, fused, st, single = ctx.state
                nadj = single_time_adjoint_steps(st["loop"]) if single else None
                lam, mu, reduced = fused.adjoint(grad.view(T, -1), st, single, nadj, comm=ode.comm)
            else:
                lam, mu = ode._adjoint_generic(ctx.state[1], ctx.state[2], grad, T)
                reduced = False
            if ode.comm is not None and not reduced:
                # the loss sums over the global batch (NCCL; the fused sweeps do it in-kernel)
                cb = ode._cb_ex
                if ctx.state[0] not in ("fused", "fused-cnf") and getattr(cb, "record_layer_events", False):
                    np_im = ode.npIM if ode.imex else 0
                    ode.comm.allreduce_sum_layered(mu, cb, np_im)
                else:
                    ode.comm.allreduce_sum(mu)
            outs = []
            off = 0
            plist = list(ode._cb_im.params) + (list(ode._cb_ex.params) if ode._cb_ex is not ode._cb_im else [])
            for p in plist:
                outs.append(mu[off:off + p.numel()].view_as(p))
                off += p.numel()
        return (lam.view(ctx.shape), None, None) + tuple(outs)
