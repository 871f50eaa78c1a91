"""ctypes binding of csrc/libgalerkin_b200.so (the C ABI declared in include/galerkin_b200.h).

There is no CPU or eager-PyTorch fallback: if the shared library is missing, or a tensor is
not an fp32 CUDA tensor, the call raises.  The handle is module-level (never stored on an
nn.Module) so modules stay picklable / deep-copyable like the reference's.
"""
import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GB200_LIB", os.path.join(_HERE, "csrc", "libgalerkin_b200.so"))   # override: tuning builds

_lock = threading.Lock()
_lib = None

c_int, c_ll, c_float, c_vp, c_sz, c_ull = (ctypes.c_int, ctypes.c_longlong, ctypes.c_float,
                                            ctypes.c_void_p, ctypes.c_size_t, ctypes.c_ulonglong)


class HeadOperand(ctypes.Structure):
    """mirror of gb200_head_operand"""
    _fields_ = [("ptr", c_vp), ("ld", c_int), ("col0", c_int), ("augmented", c_int),
                ("gamma", c_vp), ("beta", c_vp)]


_HOP = ctypes.POINTER(HeadOperand)


class EncoderParams(ctypes.Structure):
    """mirror of gb200_encoder_params (include/galerkin_b200.h)"""
    _fields_ = [(k, c_vp) for k in ("wq", "wk", "wv", "bq", "bk", "bv")] + \
               [("gamma_k", c_vp * 8), ("beta_k", c_vp * 8), ("gamma_v", c_vp * 8), ("beta_v", c_vp * 8)] + \
               [(k, c_vp) for k in ("wfc", "bfc", "w1", "b1", "w2", "b2")] + \
               [(k, c_int) for k in ("d_model", "n_head", "pos_dim", "d_ff")]


_ENCP = ctypes.POINTER(EncoderParams)


class WgradProblem(ctypes.Structure):
    """mirror of gb200_wgrad_problem"""
    _fields_ = [("G", c_vp), ("ldg", c_int), ("X", c_vp), ("ldx", c_int), ("dW", c_vp), ("ldw", c_int), ("M", c_int),
                ("N", c_int), ("T", c_ll)]

# name -> (restype, argtypes); must list every symbol of include/galerkin_b200.h
SIGNATURES = {
    "gb200_version": (c_int, []),
    "gb200_last_error": (ctypes.c_char_p, []),
    "gb200_launch_count": (c_ull, []),
    "gb200_set_rng_offset_ptr": (c_int, [c_vp]),
    "gb200_pack": (c_int, [c_int, c_vp, ctypes.POINTER(c_vp), ctypes.POINTER(c_ll), c_int, c_vp]),
    "gb200_gemm_workspace_bytes": (c_sz, [c_int] * 5),
    "gb200_gemm_suggest_ksplit": (c_int, [c_int] * 4),
    "gb200_gemm": (c_int, [c_int, c_vp, c_int, c_int, c_vp, c_int, c_int, c_vp, c_int, c_int, c_int, c_int,
                           c_int, c_ll, c_ll, c_ll, c_float, c_vp, c_int, c_vp, c_int, c_float, c_ull,
                           c_vp, c_int, c_float, c_int, c_int, c_vp, c_sz, c_vp]),
    "gb200_gemm_tc_supported": (c_int, [c_vp, c_int, c_vp, c_int, c_int, c_int, c_int]),
    "gb200_gemm_tc_suggest_ksplit": (c_int, [c_int] * 3),
    "gb200_gemm_tc_wgrad_group_workspace_bytes": (c_sz, [c_int, ctypes.POINTER(WgradProblem)]),
    "gb200_gemm_tc_wgrad_group": (c_int, [c_int, c_int, ctypes.POINTER(WgradProblem), c_vp, c_sz, c_vp]),
    "gb200_gemm_tc_set_trace": (c_int, [c_vp]),
    "gb200_gemm_tc": (c_int, [c_int, c_vp, c_int, c_int, c_vp, c_int, c_int, c_vp, c_int, c_int, c_int, c_int,
                              c_float, c_vp, c_int, c_vp, c_int, c_float, c_ull, c_vp, c_int, c_float, c_int,
                              c_int, c_vp, c_sz, c_int, c_vp]),
    "gb200_gemm_tc_gated": (c_int, [c_int, c_vp, c_int, c_int, c_vp, c_int, c_int, c_vp, c_int, c_int, c_int, c_int, c_float, c_float,
                                    c_ull, c_float, c_vp, c_int, c_int, c_int, c_vp, c_sz, c_int, c_vp]),
    "gb200_gemm_gated": (c_int, [c_int, c_vp, c_int, c_int, c_vp, c_int, c_int, c_vp, c_int, c_int, c_int, c_int, c_float, c_float,
                                    c_ull, c_float, c_vp, c_int, c_int, c_int, c_vp, c_sz, c_vp]),
    "gb200_colsum_workspace_bytes": (c_sz, [c_ll, c_int]),
    "gb200_colsum": (c_int, [c_int, c_vp, c_int, c_ll, c_int, c_float, c_int, c_vp, c_vp, c_sz, c_vp]),
    "gb200_epilogue_bwd": (c_int, [c_int, c_vp, c_int, c_vp, c_int, c_vp, c_int, c_vp, c_int, c_ll, c_int,
                                   c_int, c_float, c_float, c_ull, c_vp]),
    "gb200_epilogue_bwd_bias_workspace_bytes": (c_sz, [c_ll, c_int]),
    "gb200_epilogue_bwd_bias": (c_int, [c_int, c_vp, c_int, c_vp, c_int, c_vp, c_int, c_vp, c_int, c_ll, c_int,
                                        c_int, c_float, c_float, c_ull, c_vp, c_vp, c_sz, c_vp]),
    "gb200_layernorm_fwd": (c_int, [c_int, c_vp, c_ll, c_int, c_vp, c_vp, c_float, c_vp, c_vp, c_vp, c_vp]),
    "gb200_layernorm_bwd_workspace_bytes": (c_sz, [c_ll, c_int]),
    "gb200_layernorm_bwd": (c_int, [c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_ll, c_int, c_vp, c_vp, c_vp,
                                    c_int, c_vp, c_sz, c_vp]),
    "gb200_headnorm_fwd": (c_int, [c_int, c_vp, c_int, c_int, c_int, c_ll, c_int, c_int, c_float, c_vp, c_vp, c_vp]),
    "gb200_headnorm_bwd_workspace_bytes": (c_sz, [c_ll, c_int, c_int]),
    "gb200_headnorm_bwd": (c_int, [c_int, c_vp, c_int, c_int, c_int, c_vp, c_int, c_int, c_int, c_vp, c_vp, c_vp,
                                   c_vp, c_ll, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_sz, c_vp]),
    "gb200_attn_suggest_nsplit": (c_int, [c_int] * 3),
    "gb200_attn_xty_workspace_bytes": (c_sz, [c_int] * 4),
    "gb200_attn_xty": (c_int, [c_int, _HOP, _HOP, c_vp, c_int, c_int, c_int, c_int, c_int, c_float, c_vp, c_float,
                               c_ull, c_vp, c_int, c_vp, c_sz, c_int, c_vp]),
    "gb200_interp_bilinear_fwd": (c_int, [c_int, c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, c_int, c_vp]),
    "gb200_interp_bilinear_bwd": (c_int, [c_int, c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, c_int, c_vp]),
    "gb200_weighted_l2_loss2d_workspace_bytes": (c_sz, [c_int, c_int]),
    "gb200_weighted_l2_loss2d": (c_int, [c_int, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_float, c_float, c_float, c_float,
                                         c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "gb200_adam_clip_step_workspace_bytes": (c_sz, [c_ll]),
    "gb200_adam_clip_step": (c_int, [c_int, c_vp, c_vp, c_vp, c_vp, c_ll, c_vp, c_float, c_float, c_float, c_float, c_vp,
                                     c_vp, c_sz, c_vp]),
    "gb200_philox_scale": (c_int, [c_int, c_vp, c_ll, c_float, c_ull, c_vp]),
    "gb200_attn_xm": (c_int, [c_int, _HOP, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_vp,
                              c_int, c_int, c_int, c_float, c_int, c_vp]),
    "gb200_fourier_quad_fwd": (c_int, [c_int, _HOP, _HOP, _HOP, c_vp, c_int, c_int, c_int, c_int, c_int, c_float, c_vp,
                                       c_float, c_ull, c_vp, c_vp, c_vp]),
    "gb200_fourier_quad_bwd": (c_int, [c_int, _HOP, _HOP, _HOP, _HOP, c_vp, c_int, c_int, c_int, c_int, c_int, c_float,
                                       c_vp, c_float, c_ull, c_vp, c_int, c_int, c_int, c_int, c_vp]),
    "gb200_spectral_suggest_ysplit": (c_int, [c_ll, c_int, c_int]),
    "gb200_spectral_ydft_workspace_bytes": (c_sz, [c_ll, c_int, c_int, c_int]),
    "gb200_spectral_ydft": (c_int, [c_int, c_vp, c_ll, c_int, c_int, c_int, c_vp, c_float, c_int, c_vp,
                                    c_int, c_vp, c_sz, c_int, c_vp]),
    "gb200_spectral_xdft": (c_int, [c_int, c_vp, c_int, c_int, c_int, c_int, c_vp, c_float, c_int, c_vp,
                                    c_vp]),
    "gb200_spectral_mix_fwd": (c_int, [c_int, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_vp,
                                       c_vp]),
    "gb200_spectral_mix_bwd": (c_int, [c_int, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int,
                                       c_vp, c_vp, c_vp, c_int, c_vp]),
    "gb200_spectral_yidft_epilogue": (c_int, [c_int, c_vp, c_ll, c_int, c_int, c_int, c_vp, c_float, c_int,
                                              c_vp, c_int, c_vp, c_vp, c_int, c_vp, c_vp, c_int, c_vp]),
    "gb200_encoder_supported": (c_int, [c_int] * 4),
    "gb200_encoder_set_trace": (c_int, [c_vp]),
    "gb200_encoder_pack_bytes": (c_sz, [c_int] * 4),
    "gb200_encoder_pack": (c_int, [c_int, _ENCP, c_vp, c_vp]),
    "gb200_encoder_workspace_bytes": (c_sz, [c_int] * 5),
    "gb200_encoder_layer_fwd": (c_int, [c_int, c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp, c_int, c_int, c_int, c_float,
                                        c_float, c_vp, c_float, c_ull, c_float, c_ull, c_float, c_float, c_ull, c_float,
                                        c_ull, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_int, c_vp]),
    "gb200_encoder_bwd_workspace_bytes": (c_sz, [c_int] * 5),
    "gb200_encoder_bwd_set_trace": (c_int, [c_vp]),
    "gb200_encoder_layer_bwd": (c_int, [c_int, c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp, c_int, c_int, c_int, c_float,
                                        c_vp, c_float, c_ull, c_float, c_ull, c_float, c_float, c_float, c_ull,
                                        c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz,
                                        c_int, c_vp]),
    "gb200_conv3x3_supported": (c_int, [c_int, c_int]),
    "gb200_conv3x3_pack_bytes": (c_sz, [c_int, c_int, c_int]),
    "gb200_conv3x3_pack": (c_int, [c_int, c_vp, c_int, c_int, c_int, c_vp, c_vp]),
    "gb200_conv_split": (c_int, [c_int, c_vp, c_int, c_int, c_int, c_ll, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_float, c_ull,
                                 c_vp, c_vp]),
    "gb200_conv3x3": (c_int, [c_int, c_vp, c_vp, c_int, c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, c_int, c_vp, c_vp, c_int,
                              c_int, c_int, c_float, c_ull, c_vp]),
    "gb200_conv1_fwd": (c_int, [c_int, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_float, c_ull, c_vp]),
    "gb200_conv1_bwd_workspace_bytes": (c_sz, [c_int]),
    "gb200_conv1_bwd": (c_int, [c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_float, c_vp, c_sz,
                                c_vp]),
}


def load():
    """Load (once) and return the shared library; raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f"{LIB_PATH} not found: the sm_100a CUDA extension is not built "
                    "(run `python -c 'import __graft_entry__ as g; g.build()'`). "
                    "galerkin_transformer_b200 has no CPU / eager fallback.")
            lib = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype, fn.argtypes = res, args
            _lib = lib
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = load().gb200_last_error().decode(errors="replace")
        raise RuntimeError(f"libgalerkin_b200 {what}: {msg} (code {rc})")


def launch_count():
    return int(load().gb200_launch_count())


def require_cuda_f32(*tensors):
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("galerkin_transformer_b200 operators run on sm_100a CUDA tensors only "
                               f"(got a {t.device} tensor); there is no CPU fallback")
        if t.dtype != torch.float32:
            raise RuntimeError(f"galerkin_transformer_b200 operators are fp32 (got {t.dtype})")


def ptr(t):
    return None if t is None else t.data_ptr()


def stream_of(t):
    return torch.cuda.current_stream(t.device).cuda_stream


def workspace(nbytes, like):
    """Caller-owned scratch from PyTorch's caching allocator (stream-ordered, graph-safe)."""
    if nbytes <= 0:
        return None
    return torch.empty((nbytes + 3) // 4, dtype=torch.float32, device=like.device)
