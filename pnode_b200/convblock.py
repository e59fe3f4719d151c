"""Right-hand-side evaluator for convolutional ODE blocks of the SqueezeNext kind (BASELINE config 4,
examples-pnode/models/sqnxt_PETSc.py:70-121): a chain of  relu(bn_k(conv_k(x)))  with nn.BatchNorm2d in train mode.

It plugs into the generic time stepper in place of engine.Callbacks: `f(t, u)` (the reference's evalRHSFunction,
pnode/petsc_adjoint.py:393-412) and `vjp(t, u, w)` (RHSJacShell.multTranspose, 52-82) are evaluated WITHOUT an autograd graph.

Two implementations, both on the GPU:
  * native (`self.native`, the SqueezeNext shapes: 1x1 / (1,3) / (3,1) stride-1 same convolutions, W a power of two, channels
    multiples of 4): the whole chain -- convolutions, BatchNorm statistics, BatchNorm+ReLU forward and backward, weight
    gradients -- runs in the hand-written kernels of csrc/conv_block.cu through pnode_convblock_forward / pnode_convblock_vjp
    (one C call per evaluation; no library convolution);
  * otherwise: library convolutions (ATen) + the BatchNorm+ReLU kernels of csrc/bn_relu.cu, layer by layer.
Side effects of the module are reproduced: running_mean / running_var / num_batches_tracked advance once per evaluation,
adjoint re-evaluations included (SURVEY.md H4.iv).
"""
import ctypes as C

import torch
import torch.nn as nn

from . import _lib
from .device import _stream, dtype_code
from .engine import Callbacks
from .errors import Error


def _layers(func):
    out = []
    k = 1
    while hasattr(func, "conv%d" % k) and hasattr(func, "bn%d" % k):
        out.append((getattr(func, "conv%d" % k), getattr(func, "bn%d" % k)))
        k += 1
    return out


def recognise_convblock(func, u_meta):
    """Structural match (conv1..convK / bn1..bnK and nothing else trainable, stride 1, groups 1, affine BN with running
    statistics, train mode) + numerical probe of the fused evaluator against a deep copy of the module."""
    if not isinstance(func, nn.Module) or not u_meta.is_cuda or u_meta.dim() != 4 or not func.training:
        return None
    layers = _layers(func)
    if len(layers) < 1:
        return None
    want = []
    for conv, bn in layers:
        if not isinstance(conv, nn.Conv2d) or not isinstance(bn, nn.BatchNorm2d):
            return None
        if conv.groups != 1 or conv.dilation != (1, 1) or conv.stride != (1, 1) or conv.bias is None or \
                conv.padding_mode != "zeros" or isinstance(conv.padding, str):
            return None
        if not bn.affine or not bn.track_running_stats or bn.momentum is None:
            return None
        want += [conv.weight, conv.bias, bn.weight, bn.bias]
    plist = [p for p in func.parameters() if p.requires_grad]
    if len(plist) != len(want) or any(a is not b for a, b in zip(plist, want)):
        return None
    if any(p.dtype != u_meta.dtype or p.device != u_meta.device for p in want):
        return None
    hw = u_meta.shape[2] * u_meta.shape[3]
    if (hw * u_meta.element_size()) % 16 != 0:
        return None
    import copy

    probe = copy.deepcopy(func)
    cb = ConvBlockCallbacks(copy.deepcopy(func), u_meta.shape, _probe=True)
    tf32 = torch.backends.cudnn.allow_tf32
    with torch.no_grad():
        g = torch.Generator(device="cpu").manual_seed(99)
        x = torch.randn(tuple(u_meta.shape), generator=g, dtype=torch.float64).to(u_meta)
        try:
            # the probe checks the LOGIC of the evaluator, so the library convolutions of both sides run in IEEE fp32 for
            # its duration (two TF32 algorithm choices alone differ by ~3e-3 on this block)
            torch.backends.cudnn.allow_tf32 = False
            ref = probe(0.3, x)
            got = cb.f(0.3, x.reshape(-1)).view_as(ref)
        except Exception:
            return None
        finally:
            torch.backends.cudnn.allow_tf32 = tf32
        tol = 1e-4 if u_meta.dtype == torch.float32 else 1e-9
        if ref.shape != x.shape or not torch.allclose(got, ref, rtol=tol, atol=tol):
            return None
        rm_ok = torch.allclose(cb.layers[0][1].running_mean, probe.bn1.running_mean, rtol=tol, atol=tol)
        if not rm_ok:
            return None
    return True


class ConvBlockCallbacks(Callbacks):
    NATIVE_MIN_PIXELS = 8192

    def __init__(self, func, tensor_size, _probe=False):
        super().__init__(func, tensor_size)
        self.lib = _lib.load()
        self.layers = _layers(func)
        self.code = dtype_code(self.params[0].dtype)
        cmax = max(bn.num_features for _, bn in self.layers)
        dev = self.params[0].device
        self._work = torch.empty(int(self.lib.pnode_bn_work_bytes(cmax)), dtype=torch.uint8, device=dev)
        self.launches = 0
        self.native = self.mma = False
        self._desc = None
        self._cwork = None
        picked = self._pick_evaluator(tensor_size)
        if picked is None:
            return
        from .options import Options

        self.mma, self._desc, self._act_bytes, work_bytes = picked
        self.native = True
        self._cwork = torch.empty(work_bytes, dtype=torch.uint8, device=dev)
        self._act0 = torch.empty(self._act_bytes, dtype=torch.uint8, device=dev)  # for evaluations that are not kept
        # Forward evaluations keep their activation set (z_1..z_L + batch statistics: the forward's by-product) so that the
        # adjoint stage at the same point skips the module's forward re-evaluation; bounded by a byte budget.
        self._saved = {}
        self._saved_bytes = 0
        self._save_budget = int(float(Options().getString("pnode_convblock_save_mb", "8192")) * (1 << 20))
        self.reused_activations = 0
        self._keep = True
        self._comm = None
        if self.mma:
            self._wbuf = torch.empty(int(self.lib.pnode_convmma_weight_bytes(C.byref(self._desc))), dtype=torch.uint8,
                                     device=dev)
            self._wbuf_for = None

    def _pick_evaluator(self, tensor_size):
        """(mma, descriptor, activation bytes, work bytes) of the native evaluator that takes this shape, or None: library
        convolutions."""
        from .options import Options

        off = ("0", "false", "no")
        mode = Options().getString("pnode_convblock_native", "auto")  # auto | 1 (whenever the shape is supported) | 0
        if len(self.layers) > _lib.CONV_MAX_LAYERS or len(tensor_size) != 4 or mode in off:
            return None
        # Tensor-core evaluator (csrc/conv_mma.cu, fp32 as 3xTF32) for GEMM-sized shapes: every layer at least 32 channels
        # wide (the CIFAR blocks [256,128,8,8] and [256,256,4,4]).  -pnode_convblock_mma auto | 1 (whenever supported) | 0
        mma_mode = Options().getString("pnode_convblock_mma", "auto")
        if self.params[0].dtype == torch.float32 and mma_mode not in off:
            wide = min(min(c.in_channels, c.out_channels) for c, _ in self.layers) >= 32
            if wide or mma_mode in ("1", "true", "yes", "force"):
                desc = self._make_desc()
                nact = int(self.lib.pnode_convmma_act_bytes(C.byref(desc)))
                if nact >= 0 and int(self.lib.pnode_convmma_param_count(C.byref(desc))) == self.nparams:
                    return True, desc, nact, int(self.lib.pnode_convmma_work_bytes(C.byref(desc)))
        # CUDA-core whole-chain kernels (csrc/conv_block.cu) for the SqueezeNext shapes
        desc = self._make_desc()
        nact = int(self.lib.pnode_convblock_act_bytes(C.byref(desc)))
        # The native kernels give one thread 4 pixels x 16 output channels: they need pixels to fill the machine.  The
        # last CIFAR block ([256,256,4,4]: 4096 pixels, 256 channels) is a small GEMM per layer -- measured 2.3x slower
        # than the library GEMM convolutions there (tools/time_convblock.py), 1.7x-4.2x faster on the other three.
        pixels = int(tensor_size[0]) * int(tensor_size[2]) * int(tensor_size[3])
        enough = pixels >= self.NATIVE_MIN_PIXELS or mode in ("1", "true", "yes", "force")
        if nact >= 0 and enough and int(self.lib.pnode_convblock_param_count(C.byref(desc))) == self.nparams:
            return False, desc, nact, int(self.lib.pnode_convblock_work_bytes(C.byref(desc)))
        return None

    def _make_desc(self):
        d = _lib.ConvBlockDesc()
        d.nlayers = len(self.layers)
        d.dtype = self.code
        d.N, d.H, d.W = int(self.tensor_size[0]), int(self.tensor_size[2]), int(self.tensor_size[3])
        for k, (conv, bn) in enumerate(self.layers):
            l = d.layer[k]
            l.cin, l.cout = conv.in_channels, conv.out_channels
            l.kh, l.kw = conv.kernel_size
            l.ph, l.pw = conv.padding
            l.eps, l.momentum = float(bn.eps), float(bn.momentum)
        self._refresh_pointers(d)
        return d

    def _refresh_pointers(self, d):
        """Parameters are borrowed, never copied (SURVEY.md section 8b): their addresses are re-read at the start of every
        solve / adjoint sweep (begin()), not cached across optimiser steps."""
        for k, (conv, bn) in enumerate(self.layers):
            l = d.layer[k]
            l.d_weight, l.d_bias = conv.weight.data_ptr(), conv.bias.data_ptr()
            l.d_gamma, l.d_beta = bn.weight.data_ptr(), bn.bias.data_ptr()
            l.d_running_mean, l.d_running_var = bn.running_mean.data_ptr(), bn.running_var.data_ptr()
            l.d_num_batches_tracked = bn.num_batches_tracked.data_ptr()

    def _param_versions(self):
        return tuple(p._version for p in self.params)

    def begin(self, forward, keep=True, comm=None):
        """Called by the time stepper at the start of a forward solve (forward=True; keep = an adjoint sweep will follow) and
        of an adjoint sweep.  comm: the run's BatchComm (batch sharded over GPUs) or None."""
        if not self.native:
            if comm is not None and comm.world > 1:
                raise Error(-40, "batch-sharded conv ODE blocks need the native evaluator (global BatchNorm statistics are "
                                 "exchanged inside csrc/conv_block.cu); this shape runs on library convolutions")
            return
        self._refresh_pointers(self._desc)
        if self.mma:
            self._prepare_weights()
        self._comm = comm if (comm is not None and comm.world > 1) else None
        d = self._desc
        if self._comm is not None:
            if not self._comm.enable_peer_reduce():
                raise Error(-41, "batch-sharded conv ODE blocks need NVLink peer (symmetric) memory for the BatchNorm statistics")
            if not self._comm.same_on_all_ranks(int(d.N)):
                # the in-kernel statistics exchanges are matched one to one across the ranks; a rank with a bigger shard can
                # run out of its activation budget and re-evaluate (more exchanges) where the others do not
                raise Error(-42, "batch-sharded conv ODE blocks need shards of equal size on every rank (this rank holds %d "
                                 "samples)" % int(d.N))
            d.d_peer_bufs = self._comm.peer["ptrs_dev"]
            d.rank, d.world = self._comm.rank, self._comm.world
            d.global_pixels = self._comm.global_count(int(d.N) * int(d.H) * int(d.W))
        else:
            d.d_peer_bufs, d.rank, d.world, d.global_pixels, d.epoch = None, 0, 1, 0, 0
        if forward:
            self._saved.clear()
            self._saved_bytes = 0
            self._keep = bool(keep)

    def _prepare_weights(self):
        """Weight operands (hi/lo, forward and data-gradient layouts) of the tensor-core evaluator: rewritten when a
        parameter has changed (parameters are borrowed, never cached across optimiser steps)."""
        ver = tuple((conv.weight.data_ptr(), conv.weight._version) for conv, _ in self.layers)
        if ver != self._wbuf_for:
            self._refresh_pointers(self._desc)
            _lib.check(self.lib.pnode_convmma_prepare(C.byref(self._desc), self._wbuf.data_ptr(), _stream()))
            self._wbuf_for = ver
            self.launches += len(self.layers)

    def release(self):
        super().release()
        if self.native:
            self._saved.clear()
            self._saved_bytes = 0

    def mark(self):
        super().mark()
        self._saved_mark = set(self._saved.keys()) if self.native else set()

    def rollback(self):
        """A rejected adaptive attempt: forget the activation sets its stage evaluations kept."""
        super().rollback()
        if self.native:
            for k in [k for k in self._saved if k not in getattr(self, "_saved_mark", set())]:
                del self._saved[k]
                self._saved_bytes -= self._act_bytes

    def _act_for(self, u):
        """Activation buffer for a forward evaluation at u: a kept one while the budget lasts, else the shared one."""
        if not self._keep or self._saved_bytes + self._act_bytes > self._save_budget:
            return self._act0
        act = torch.empty(self._act_bytes, dtype=torch.uint8, device=u.device)
        self._saved[u.data_ptr()] = (u, u._version, self._param_versions(), act)  # holding u keeps its address unique
        self._saved_bytes += self._act_bytes
        return act

    def _native_f(self, u, out=None, base=None, base_coef=0.0, k_coef=1.0, k=None, keep=True):
        if out is None and k is None:
            out = torch.empty_like(u)
        act = self._act_for(u) if keep else self._act0
        if self._comm is not None:
            self._desc.epoch = self._comm.reserve_epochs(len(self.layers))
        if self.mma:
            self._prepare_weights()
            _lib.check(self.lib.pnode_convmma_forward(C.byref(self._desc), self._wbuf.data_ptr(), u.data_ptr(),
                                                      None if out is None else out.data_ptr(),
                                                      None if base is None else base.data_ptr(), float(base_coef),
                                                      float(k_coef), None if k is None else k.data_ptr(), act.data_ptr(),
                                                      self._cwork.data_ptr(), _stream()))
            self.launches += 3 * len(self.layers) + 2
            return out
        _lib.check(self.lib.pnode_convblock_forward(C.byref(self._desc), u.data_ptr(), None if out is None else out.data_ptr(),
                                                    None if base is None else base.data_ptr(), float(base_coef), float(k_coef),
                                                    None if k is None else k.data_ptr(), act.data_ptr(), _stream()))
        self.launches += len(self.layers) + 1
        return out

    def _native_vjp(self, u, w, want_u, grads, coef, accumulate):
        if not w.is_contiguous():
            w = w.contiguous()
        vu = torch.empty_like(u) if want_u else None
        ent = self._saved.get(u.data_ptr())
        valid = ent is not None and ent[1] == u._version and ent[2] == self._param_versions() and ent[0].numel() == u.numel()
        act = ent[3] if valid else self._act0
        if self._comm is not None:
            self._desc.epoch = self._comm.reserve_epochs(len(self.layers) * (1 if valid else 2))
        L = len(self.layers)
        if self.mma:
            self._prepare_weights()
            _lib.check(self.lib.pnode_convmma_vjp(C.byref(self._desc), self._wbuf.data_ptr(), u.data_ptr(), w.data_ptr(),
                                                  None if vu is None else vu.data_ptr(),
                                                  None if grads is None else grads.data_ptr(), float(coef), int(accumulate),
                                                  act.data_ptr(), int(valid), self._cwork.data_ptr(), _stream()))
            self.reused_activations += int(valid)
            self.launches += (L + 1 if valid else 3 * L + 1) + 1 + L + (4 * L if grads is not None else 0) + 2 * L + 1
            return vu
        _lib.check(self.lib.pnode_convblock_vjp(C.byref(self._desc), u.data_ptr(), w.data_ptr(),
                                                None if vu is None else vu.data_ptr(),
                                                None if grads is None else grads.data_ptr(), float(coef), int(accumulate),
                                                act.data_ptr(), int(valid), self._cwork.data_ptr(), _stream()))
        self.reused_activations += int(valid)
        self.launches += (0 if valid else L) + 1 + (L if grads is not None else 0) + (L if want_u else L - 1) + \
            (1 if grads is not None else 0)
        return vu

    def f_and_combine(self, t, u, base, coef):
        """k = f(t, u) and y = base + coef * k in ONE output pass (the RK stage combination fused into the block's last
        kernel): returns (k, y).  Used by engine.GenericTS._rk_attempt when the next stage depends on k alone."""
        self.nfe += 1
        if hasattr(self.func, "nfe"):
            self.func.nfe += 1
        if not self.native:
            with torch.no_grad():
                out, _ = self._forward(t, u, save=False)
            k = out.reshape(-1)
            return k, torch.add(base, k, alpha=float(coef))
        k, y = torch.empty_like(u), torch.empty_like(u)
        self._native_f(u, out=y, base=base, base_coef=1.0, k_coef=coef, k=k)
        return k, y

    def vjp_accumulate(self, t, u, w, mu, coef):
        """vjp + `mu += coef * (df/dp)^T w` in the same call (the engine uses it when present): J^T w is returned."""
        if not self.native:
            vu, gp = self.vjp(t, u, w)
            return vu, gp
        self.nvjp += 1
        if hasattr(self.func, "nfe"):
            self.func.nfe += 1
        return self._native_vjp(u, w, True, mu, coef, True), None

    # -- one layer -----------------------------------------------------------------------------------------------
    def _bn_relu_fwd(self, z, bn):
        N, Cc, H, W = z.shape
        y = torch.empty_like(z)
        mean = torch.empty(Cc, dtype=z.dtype, device=z.device)
        invstd = torch.empty(Cc, dtype=z.dtype, device=z.device)
        _lib.check(self.lib.pnode_bn_relu_forward(z.data_ptr(), y.data_ptr(), bn.weight.data_ptr(), bn.bias.data_ptr(),
                                                  bn.running_mean.data_ptr(), bn.running_var.data_ptr(), mean.data_ptr(),
                                                  invstd.data_ptr(), N, Cc, H * W, float(bn.eps), float(bn.momentum),
                                                  self._work.data_ptr(), self.code, _stream()))
        bn.num_batches_tracked += 1
        self.launches += 2
        return y, mean, invstd

    def _forward(self, t, u, save):
        x = u.view(self.tensor_size)
        saved = []
        for conv, bn in self.layers:
            z = torch.nn.functional.conv2d(x, conv.weight, conv.bias, conv.stride, conv.padding)
            if not z.is_contiguous():
                z = z.contiguous()
            y, mean, invstd = self._bn_relu_fwd(z, bn)
            if save:
                saved.append((x, z, y, mean, invstd))
            x = y
        return x, saved

    # -- the two closures the engine needs ---------------------------------------------------------------------------
    def f(self, t, u, keep=True):
        self.nfe += 1
        if hasattr(self.func, "nfe"):
            self.func.nfe += 1
        if self.native:
            return self._native_f(u)
        with torch.no_grad():
            out, _ = self._forward(t, u, save=False)
        return out.reshape(-1)

    def vjp(self, t, u, w, want_u=True, want_params=True):
        self.nvjp += 1
        if hasattr(self.func, "nfe"):
            self.func.nfe += 1  # the reference's adjoint re-evaluates func once per stage (petsc_adjoint.py:68)
        if self.native:
            grads = torch.empty(self.nparams, dtype=u.dtype, device=u.device) if want_params else None
            vu = self._native_vjp(u, w, want_u, grads, 1.0, False)
            return vu, (list(torch.split(grads, self.sizes)) if want_params else [])
        with torch.no_grad():
            out, saved = self._forward(t, u, save=True)
            dy = w.view(out.shape)
            if not dy.is_contiguous():
                dy = dy.contiguous()
            grads = []
            for (conv, bn), (x, z, y, mean, invstd) in zip(reversed(self.layers), reversed(saved)):
                N, Cc, H, W = z.shape
                dz = torch.empty_like(z)
                dgamma = torch.empty(Cc, dtype=z.dtype, device=z.device)
                dbeta = torch.empty(Cc, dtype=z.dtype, device=z.device)
                _lib.check(self.lib.pnode_bn_relu_backward(dy.data_ptr(), z.data_ptr(), y.data_ptr(), bn.weight.data_ptr(),
                                                           mean.data_ptr(), invstd.data_ptr(), dz.data_ptr(),
                                                           dgamma.data_ptr(), dbeta.data_ptr(), N, Cc, H * W,
                                                           self._work.data_ptr(), self.code, _stream()))
                self.launches += 2
                dx, dw, db = torch.ops.aten.convolution_backward(
                    dz, x, conv.weight, [conv.out_channels], list(conv.stride), list(conv.padding), list(conv.dilation),
                    False, [0, 0], 1, [True, True, True])
                grads = [dw, db, dgamma, dbeta] + grads
                dy = dx if dx.is_contiguous() else dx.contiguous()
        vu = dy.reshape(-1) if want_u else None
        return vu, (grads if want_params else [])
