"""ctypes binding of libddrl_b200.so (C ABI: include/ddrl_b200.h).

There is no CPU or PyTorch fallback behind these calls: if the shared library is missing or
a call fails, a ``DDRLError`` is raised.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# DDRL_LIB_PATH: development override (e.g. an instrumented build); the product path is the in-tree library
LIB_PATH = os.environ.get("DDRL_LIB_PATH") or os.path.join(_HERE, "libddrl_b200.so")


class DDRLError(RuntimeError):
    pass


class NetDesc(C.Structure):
    _fields_ = [("arch", C.c_int32), ("in_ch", C.c_int32), ("act_dim", C.c_int32), ("dist", C.c_int32),
                ("shared", C.c_int32), ("feat", C.c_int32), ("gemm_mode", C.c_int32), ("laser_ch", C.c_int32)]


class PPOHparams(C.Structure):
    _fields_ = [("ppo_clip", C.c_float), ("dual_clip", C.c_float), ("v_coef", C.c_float), ("ent_coef", C.c_float),
                ("max_grad_norm", C.c_float), ("clip_grad", C.c_int32), ("smooth_l1", C.c_int32),
                ("lr", C.c_float), ("lr_actor", C.c_float), ("lr_critic", C.c_float),
                ("beta1", C.c_float), ("beta2", C.c_float), ("adam_eps", C.c_float),
                ("value_clip", C.c_float), ("ppo_stats", C.c_int32)]


class GatherJob(C.Structure):
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("row_bytes", C.c_int64), ("src_stride", C.c_int64),
                ("dst_stride", C.c_int64), ("src_rows", C.c_int64)]


GATHER_MAX_JOBS = 12       # DDRL_GATHER_MAX_JOBS


class ConvDesc(C.Structure):
    _fields_ = [(k, C.c_int32) for k in ("B", "H", "W", "Cin", "Cout", "KH", "KW", "stride", "pad")]


ARCH = {"atari": 0, "nav": 1, "navped": 2, "nav1d": 3, "mlp": 4}
DIST = {"categorical": 0, "gaussian": 1}
GEMM_MODE = {"simt": 0, "tc": 1, "tc2": 2, "tc3": 3}

_P = C.c_void_p
_I = C.c_int
_F = C.c_float
_L = C.c_int64

# name -> (restype, argtypes): every symbol include/ddrl_b200.h declares
SIGNATURES = {
    "ddrl_version": (_I, []),
    "ddrl_error_string": (C.c_char_p, [_I]),
    "ddrl_last_cuda_error": (C.c_char_p, []),
    "ddrl_launch_count": (_L, []),
    "ddrl_launch_count_reset": (None, []),
    "ddrl_prof_start": (_I, [_P]),
    "ddrl_prof_stop": (_I, [C.c_char_p, _I]),
    "ddrl_gae_f32": (_I, [_P, _P, _P, C.POINTER(_F), _F, _I, _I, _I, _P, _P, _I, _P]),
    "ddrl_gae_tempo": (_I, [_P, _P, _P, _P, C.POINTER(C.c_double), _I, C.c_double, _I, _I, _I, _P, _P, _I, _P]),
    "ddrl_easybytes_decode": (_I, [_P, _P, _I, C.c_uint, _P, _P]),
    "ddrl_easybytes_reply_bytes": (_L, [_I, _I, _I]),
    "ddrl_easybytes_encode_replies": (_I, [_P, _I, _P, _P, _I, _I, _I, _I, _P, _P]),
    "ddrl_sample_categorical_probs": (_I, [_P, _I, _P, _I, _I, _P, _P, _P]),
    "ddrl_categorical_head": (_I, [_P, _I, _P, _I, _I, _P, _P, _P, _P]),
    "ddrl_gaussian_head": (_I, [_P, _I, _P, _P, _I, _I, _P, _P, _P]),
    "ddrl_ppo_loss_categorical": (_I, [_P, _I, _P, _P, _P, _P, _P, _I, _I, _F, C.POINTER(PPOHparams), _I, _P, _I, _P, _P, _P]),
    "ddrl_ppo_loss_gaussian": (_I, [_P, _I, _P, _P, _P, _P, _P, _P, _I, _I, _F, C.POINTER(PPOHparams), _I, _P, _I, _P, _P, _P, _P]),
"ddrl_ppo_loss_categorical_v": (_I, [_P, _I, _P, _P, _P, _P, _P, _I, _I, _F, C.POINTER(PPOHparams), _I, _P, _I, _P, _P, _P, _P,
                                        _P]),
    "ddrl_ppo_loss_gaussian_v": (_I, [_P, _I, _P, _P, _P, _P, _P, _P, _I, _I, _F, C.POINTER(PPOHparams), _I, _P, _I, _P, _P, _P, _P,
                                     _P, _P]),
    "ddrl_adv_moments": (_I, [_P, _I, _P, _P]),
    "ddrl_adv_normalize": (_I, [_P, _I, _P, _F, _P, _P]),
    "ddrl_obs_moments_ws_bytes": (_L, [_I, _I]),
    "ddrl_obs_moments": (_I, [_P, _I, _I, _P, _P, _P, _L, _P]),
    "ddrl_obs_rms_update": (_I, [_P, _P, _P, _P, C.c_double, _I, _P, _P, _P]),
    "ddrl_obs_normalize": (_I, [_P, _I, _I, _P, _P, _F, _P, _P]),
    "ddrl_value_loss": (_I, [_P, _P, _I, _F, C.POINTER(PPOHparams), _I, _P, _P, _P]),
    "ddrl_clip_adam": (_I, [_P, _P, _P, _P, _L, C.POINTER(_L), C.POINTER(_F), _I, _I, C.POINTER(PPOHparams), _P, _P]),
    "ddrl_gemm_f32": (_I, [_I, _I, _I, _I, _I, _P, _I, _P, _I, _P, _I, _P, _I, _I, _P]),
    "ddrl_conv_nhwc_f32": (_I, [_I, _I, C.POINTER(ConvDesc), _P, _P, _P, _P, _I, _P, _P, _P]),
    "ddrl_net_create": (_I, [C.POINTER(NetDesc), C.POINTER(_P)]),
    "ddrl_net_destroy": (_I, [_P]),
    "ddrl_net_num_tensors": (_I, [_P]),
    "ddrl_net_num_params": (_L, [_P]),
    "ddrl_net_tensor_info": (_I, [_P, _I, C.c_char_p, _I, C.POINTER(_L), C.POINTER(_I), C.POINTER(_L)]),
    "ddrl_net_bind": (_I, [_P, _P, _P, _P, _P]),
    "ddrl_net_params_changed": (_I, [_P]),
    "ddrl_net_set_extra_critics": (_I, [_P, _I, C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.POINTER(_I)]),
    "ddrl_net_num_obs": (_I, [_P]),
    "ddrl_net_obs_elems": (_L, [_P, _I]),
    "ddrl_net_forward": (_I, [_P, C.POINTER(_P), _I, _I, _P, _P, _P, _P, _P, _P]),
    "ddrl_net_encode": (_I, [_P, C.POINTER(_P), _I, _I, _I, _P, _P]),
    "ddrl_net_backward": (_I, [_P, C.POINTER(_P), _I, _I, _I, _P, _P, _P, _P, C.POINTER(PPOHparams), _I, _P]),
    "ddrl_net_backward_v": (_I, [_P, C.POINTER(_P), _I, _I, _I, _P, _P, _P, _P, _P, C.POINTER(PPOHparams), _I, _P]),
    "ddrl_net_backward_segment": (_I, [_P, C.POINTER(_P), _I, _I, _I, _P, _P, _P, _P, C.POINTER(PPOHparams), _I, _I, C.POINTER(_I), _P]),
    "ddrl_net_tensor_segment": (_I, [_P, _I]),
    "ddrl_net_backward_minibatch": (_I, [_P, C.POINTER(_P), _I, _I, _I, _P, _P, _P, _P, C.POINTER(PPOHparams), _P]),
    "ddrl_net_backward_minibatch_v": (_I, [_P, C.POINTER(_P), _I, _I, _I, _P, _P, _P, _P, _P, C.POINTER(PPOHparams), _P]),
    "ddrl_gather_rows": (_I, [_P, _I, C.POINTER(GatherJob), _I, _P]),
    "ddrl_set_deterministic": (_I, [_I]),
    "ddrl_peer_allreduce_flag_bytes": (_I, []),
    "ddrl_peer_allreduce_f32": (_I, [C.POINTER(_P), _P, C.POINTER(_P), _I, _I, C.c_int64, C.c_int64, C.c_uint32, _P]),
    "ddrl_net_clip_adam": (_I, [_P, _I, C.POINTER(PPOHparams), _P, _P]),
    "ddrl_net_workspace_bytes": (_L, [_P]),
}

_lib = None


def load():
    """Loads the shared library (once).  Raises DDRLError if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DDRLError(
            "libddrl_b200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` or "
            "`make -C ddrl4nav_b200/csrc`. There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError => ABI mismatch, fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(code, what=""):
    if code != 0:
        lib = load()
        msg = lib.ddrl_error_string(code).decode()
        if code == -2:
            msg += ": " + lib.ddrl_last_cuda_error().decode()
        raise DDRLError("%s failed (%d): %s" % (what or "ddrl call", code, msg))


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def current_stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise DDRLError("ddrl4nav_b200 kernels need CUDA tensors (no CPU fallback); got device %s" % t.device)
