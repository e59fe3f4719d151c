"""ctypes binding of include/pnode_b200.h.  There is NO fallback: if the shared library is missing or a symbol is
absent, importing the engine fails loudly (the product path never runs on the CPU)."""
import ctypes as C
import os

from .errors import Error

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PNODE_B200_LIB") or os.path.join(_HERE, "csrc", "libpnode_b200.so")  # env: tuning builds only

F32, F64 = 0, 1
MAX_TERMS, MAX_STAGES, MAX_SRCS = 16, 7, 32
SEG_COEF, SEG_NEG, SEG_RSQRT = 0, 1, 2


class RKTableau(C.Structure):
    _fields_ = [("s", C.c_int32), ("fsal", C.c_int32), ("a", (C.c_double * MAX_STAGES) * MAX_STAGES),
                ("b", C.c_double * MAX_STAGES), ("c", C.c_double * MAX_STAGES), ("be", C.c_double * MAX_STAGES),
                ("has_be", C.c_int32), ("order", C.c_int32)]


class MlpDesc(C.Structure):
    _fields_ = [("dim", C.c_int32), ("hidden", C.c_int32), ("phi", C.c_int32), ("dtype", C.c_int32),
                ("d_w1", C.c_void_p), ("d_b1", C.c_void_p), ("d_w2", C.c_void_p), ("d_b2", C.c_void_p)]


class CnfDesc(C.Structure):
    _fields_ = [("dim", C.c_int32), ("hidden", C.c_int32), ("dtype", C.c_int32), ("t_via_f32", C.c_int32)] + \
               [(n, C.c_void_p) for n in ("d_w1", "d_b1", "d_hb1", "d_hgw1", "d_hgb1", "d_w2", "d_b2", "d_hb2", "d_hgw2",
                                          "d_hgb2", "d_e")]


CTL_MAX_SPAN = 16
CTL_MAX_LOG = 1024


class Step(C.Structure):
    _fields_ = [("t", C.c_double), ("h", C.c_double), ("out_slot", C.c_int32), ("in_slot", C.c_int32)]


class CnfCtl(C.Structure):
    """include/pnode_b200.h: pnode_cnf_ctl (the device-resident step controller's state and attempt log)."""
    _fields_ = [("t", C.c_double), ("h", C.c_double), ("t_end", C.c_double), ("dt_span_cached", C.c_double),
                ("span", C.c_double * CTL_MAX_SPAN), ("n_global", C.c_double), ("delta", C.c_double)] + \
               [(n, C.c_int32) for n in ("nspan", "order", "max_reject", "done", "cur", "kcur", "have_k", "steps",
                                         "attempts", "rejections", "prev_ok", "ctr", "cur_sol_index", "pending_slot",
                                         "max_steps", "single", "prev_out_slot")] + \
               [("sumsq", C.c_double), ("epoch_next", C.c_uint64), ("log_t", C.c_double * CTL_MAX_LOG), ("log_h", C.c_double * CTL_MAX_LOG),
                ("log_enorm", C.c_double * CTL_MAX_LOG), ("log_accepted", C.c_int32 * CTL_MAX_LOG),
                ("sched", Step * CTL_MAX_LOG)]


CONV_MAX_LAYERS = 8
DMLP_MAX_LAYERS = 8
CIRC_MAX_TAPS = 16


class DmlpDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("nlayers", "dtype", "batch", "reserved")] + \
               [("dims", C.c_int32 * (DMLP_MAX_LAYERS + 1)), ("d_weight", C.c_void_p * DMLP_MAX_LAYERS),
                ("d_bias", C.c_void_p * DMLP_MAX_LAYERS), ("mu_w_off", C.c_int64 * DMLP_MAX_LAYERS),
                ("mu_b_off", C.c_int64 * DMLP_MAX_LAYERS), ("out_scale", C.c_double)]


class CnfNetDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("nlayers", "dtype", "batch", "t_f32")] + \
               [("dims", C.c_int32 * (DMLP_MAX_LAYERS + 1))] + \
               [(n, C.c_void_p * DMLP_MAX_LAYERS) for n in ("d_weight", "d_bias", "d_hyper_bias", "d_gate_weight",
                                                            "d_gate_bias")] + \
               [(n, C.c_int64 * DMLP_MAX_LAYERS) for n in ("mu_w_off", "mu_b_off", "mu_hbw_off", "mu_hgw_off",
                                                          "mu_hgb_off")] + [("d_e", C.c_void_p), ("trace", C.c_int32)]


class ConvLayer(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("cin", "cout", "kh", "kw", "ph", "pw")] + \
               [(n, C.c_void_p) for n in ("d_weight", "d_bias", "d_gamma", "d_beta", "d_running_mean", "d_running_var",
                                          "d_num_batches_tracked")] + [("eps", C.c_double), ("momentum", C.c_double)]


class ConvBlockDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("nlayers", "dtype", "N", "H", "W", "reserved")] + \
               [("layer", ConvLayer * CONV_MAX_LAYERS), ("d_peer_bufs", C.c_void_p), ("rank", C.c_int32), ("world", C.c_int32),
                ("epoch", C.c_uint64), ("global_pixels", C.c_int64)]


_vp, _i, _i64, _d = C.c_void_p, C.c_int, C.c_int64, C.c_double
_SIGNATURES = {
    "pnode_abi_version": (C.c_int, []),
    "pnode_last_error": (C.c_char_p, []),
    "pnode_device_sm_count": (C.c_int, [C.POINTER(C.c_int)]),
    "pnode_lincomb": (C.c_int, [_vp, _vp, _d, C.POINTER(_vp), C.POINTER(_d), _i, _i64, _i, _vp]),
    "pnode_wrms_work_bytes": (_i64, []),
    "pnode_rk_complete_wrms": (C.c_int, [_vp, _vp, C.POINTER(_vp), C.POINTER(_d), C.POINTER(_d), _i, _i64, _d, _d, _vp,
                                         _vp, _i, _vp]),
    "pnode_multi_axpy": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_i64), _i, _d, _i, _vp]),
    "pnode_mdot_work_bytes": (_i64, []),
    "pnode_mdot": (C.c_int, [_vp, C.POINTER(_vp), _i, _vp, _i64, _vp, _i, _vp]),
    "pnode_mdot_seg": (C.c_int, [_vp, _vp, _i, _vp, _i64, _i64, _i, _vp]),
    "pnode_lincomb_seg": (C.c_int, [_vp, _vp, _d, _vp, _vp, _i, _i, _i64, _i64, _i, _vp]),
    "pnode_mlp_rk_supported": (C.c_int, [_i, _i, _i, _i, _i]),
    "pnode_mlp_rk_forward": (C.c_int, [C.POINTER(MlpDesc), C.POINTER(RKTableau), _vp, _i64, _vp, _i, _vp, _vp, _vp]),
    "pnode_mlp_rk_ckpt_rows": (C.c_int, [C.POINTER(MlpDesc), C.POINTER(RKTableau)]),
    "pnode_mlp_rk_adjoint_work_bytes": (_i64, [C.POINTER(MlpDesc)]),
    "pnode_mlp_rk_adjoint": (C.c_int, [C.POINTER(MlpDesc), C.POINTER(RKTableau), _i64, _vp, _i, _i, _vp, _vp, _vp, _vp,
                                       _vp, _vp]),
    "pnode_mlp_rk_forward_so": (C.c_int, [C.POINTER(MlpDesc), C.POINTER(RKTableau), _vp, _i64, _vp, _i, _vp, _vp, _vp]),
    "pnode_mlp_rk_adjoint_so": (C.c_int, [C.POINTER(MlpDesc), C.POINTER(RKTableau), _i64, _vp, _i, _i, _vp, _vp, _vp, _vp,
                                          _vp, _vp, _i, _i, C.c_uint64, _vp]),
    "pnode_cnf_rk_supported": (C.c_int, [_i, _i, _i, _i]),
    "pnode_cnf_rk_attempt": (C.c_int, [C.POINTER(CnfDesc), C.POINTER(RKTableau), _vp, _vp, _i64, _d, _d, _vp, _vp, _vp, _d,
                                       _d, _vp, _vp, _vp]),
    "pnode_cnf_rk_attempts_ctl": (C.c_int, [C.POINTER(CnfDesc), C.POINTER(RKTableau), _vp, _vp, _i64, _vp, _i64, _vp, _d, _d,
                                            _vp, _vp, _i, _vp]),
    "pnode_cnf_rk_solve_ctl": (C.c_int, [C.POINTER(CnfDesc), C.POINTER(RKTableau), _vp, _vp, _i64, _vp, _i64, _vp, _d, _d,
                                         _vp, _vp, _vp]),
    "pnode_cnf_rk_solve_ctl_dp": (C.c_int, [C.POINTER(CnfDesc), C.POINTER(RKTableau), _vp, _vp, _i64, _vp, _i64, _vp, _d, _d,
                                            _vp, _vp, _vp, _i, _i, _vp]),
    "pnode_cnf_ctl_probe": (C.c_int, [_vp, _vp, _i, _vp]),
    "pnode_cnf_rk_gather_ctl": (C.c_int, [_vp, _vp, _vp, _vp, _i, _i64, _i, _vp]),
    "pnode_cnf_rk_adjoint_ctl": (C.c_int, [C.POINTER(CnfDesc), C.POINTER(RKTableau), _i64, _vp, _i, _vp, _vp, _vp, _vp, _vp,
                                           _vp]),
    "pnode_cnf_rk_adjoint_work_bytes": (_i64, [C.POINTER(CnfDesc)]),
    "pnode_cnf_rk_adjoint": (C.c_int, [C.POINTER(CnfDesc), C.POINTER(RKTableau), _i64, _vp, _i, _i, _vp, _vp, _vp, _vp,
                                       _vp, _vp]),
    "pnode_bn_work_bytes": (_i64, [_i]),
    "pnode_bn_relu_forward": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _d, _d, _vp, _i, _vp]),
    "pnode_bn_relu_backward": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _i, _vp]),
    "pnode_convblock_act_bytes": (_i64, [C.POINTER(ConvBlockDesc)]),
    "pnode_convblock_work_bytes": (_i64, [C.POINTER(ConvBlockDesc)]),
    "pnode_convblock_param_count": (_i64, [C.POINTER(ConvBlockDesc)]),
    "pnode_convblock_forward": (C.c_int, [C.POINTER(ConvBlockDesc), _vp, _vp, _vp, _d, _d, _vp, _vp, _vp]),
    "pnode_convblock_vjp": (C.c_int, [C.POINTER(ConvBlockDesc), _vp, _vp, _vp, _vp, _d, _i, _vp, _i, _vp, _vp]),
    "pnode_convmma_act_bytes": (_i64, [C.POINTER(ConvBlockDesc)]),
    "pnode_convmma_work_bytes": (_i64, [C.POINTER(ConvBlockDesc)]),
    "pnode_convmma_weight_bytes": (_i64, [C.POINTER(ConvBlockDesc)]),
    "pnode_convmma_param_count": (_i64, [C.POINTER(ConvBlockDesc)]),
    "pnode_convmma_prepare": (C.c_int, [C.POINTER(ConvBlockDesc), _vp, _vp]),
    "pnode_convmma_forward": (C.c_int, [C.POINTER(ConvBlockDesc), _vp, _vp, _vp, _vp, _d, _d, _vp, _vp, _vp, _vp]),
    "pnode_convmma_vjp": (C.c_int, [C.POINTER(ConvBlockDesc), _vp, _vp, _vp, _vp, _vp, _d, _i, _vp, _i, _vp, _vp]),
    "pnode_peer_buffer_bytes": (_i64, [_i]),
    "pnode_mlp_rk_adjoint_dp": (C.c_int, [C.POINTER(MlpDesc), C.POINTER(RKTableau), _i64, _vp, _i, _i, _vp, _vp, _vp, _vp,
                                          _vp, _vp, _i, _i, C.c_uint64, _vp]),
    "pnode_cnf_rk_adjoint_dp": (C.c_int, [C.POINTER(CnfDesc), C.POINTER(RKTableau), _i64, _vp, _i, _i, _vp, _vp, _vp, _vp,
                                          _vp, _vp, _i, _i, C.c_uint64, _vp]),
    "pnode_sliced_bytes": (_i64, [_i, _i, _i]),
    "pnode_slice_rows": (C.c_int, [_i, _vp, _i64, _i, _i, _vp, _vp, _vp]),
    "pnode_slice_cols": (C.c_int, [_i, _vp, _i64, _i, _i, _vp, _vp, _vp, _d, _vp]),
    "pnode_sliced_gemm": (C.c_int, [_i, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _i64, _d, _vp, _i, _vp, _i64, _i, _vp]),
    "pnode_dmlp_weight_bytes": (_i64, [C.POINTER(DmlpDesc)]),
    "pnode_dmlp_act_bytes": (_i64, [C.POINTER(DmlpDesc)]),
    "pnode_dmlp_work_bytes": (_i64, [C.POINTER(DmlpDesc)]),
    "pnode_dmlp_prepare": (C.c_int, [C.POINTER(DmlpDesc), _vp, _vp]),
    "pnode_dmlp_forward": (C.c_int, [C.POINTER(DmlpDesc), _vp, _vp, _vp, _vp, _vp, _vp]),
    "pnode_dmlp_vjp": (C.c_int, [C.POINTER(DmlpDesc), _vp, _vp, _vp, _vp, _vp, _d, _vp, _vp]),
    "pnode_dmlp_vjp_ev": (C.c_int, [C.POINTER(DmlpDesc), _vp, _vp, _vp, _vp, _vp, _d, _vp, _vp, _vp]),
    "pnode_cnfnet_weight_bytes": (_i64, [C.POINTER(CnfNetDesc)]),
    "pnode_cnfnet_act_bytes": (_i64, [C.POINTER(CnfNetDesc)]),
    "pnode_cnfnet_work_bytes": (_i64, [C.POINTER(CnfNetDesc)]),
    "pnode_cnfnet_prepare": (C.c_int, [C.POINTER(CnfNetDesc), _vp, _vp]),
    "pnode_cnfnet_forward": (C.c_int, [C.POINTER(CnfNetDesc), _vp, _d, _vp, _vp, _vp, _vp, _vp]),
    "pnode_cnfnet_vjp": (C.c_int, [C.POINTER(CnfNetDesc), _vp, _d, _vp, _vp, _vp, _vp, _d, _vp, _vp]),
    "pnode_circulant_apply":(C.c_int, [_vp, _vp, _i, _i, C.POINTER(C.c_int32), C.POINTER(_d), _i, _i, _i, _vp]),
    "pnode_circulant_work_bytes": (_i64, [_i]),
    "pnode_circulant_inverse": (C.c_int, [_vp, _i, _d, _vp, _i, _vp, _vp]),
    "pnode_peak_fma": (C.c_int, [_i, _i, C.POINTER(_d), C.POINTER(C.c_float)]),
    "pnode_tanh_probe": (C.c_int, [_vp, _vp, _i64, _i, _vp]),
    "pnode_acc128_probe": (C.c_int, [_vp, _i64, _vp, _vp, _vp]),
}

_lib = None


def load():
    """Load (once) and type the library.  Raises pnode_b200.Error if it is missing: build it with
    `python -m pnode_b200.build` (or __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise Error(-1, "native library %s not built; run `python -m pnode_b200.build`. "
                        "There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            raise Error(-2, "native library %s lacks symbol %s (stale build?)" % (LIB_PATH, name))
        fn.restype = res
        fn.argtypes = args
    if lib.pnode_abi_version() != 1:
        raise Error(-3, "ABI version mismatch")
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise Error(rc, load().pnode_last_error().decode("utf-8", "replace"))


def exported_symbols():
    return sorted(_SIGNATURES)
