"""ctypes binding of libmfm_b200.so (the C-ABI declared in include/mfm_b200.h).

torch is used only for device memory and streams; every pointer handed to the library is a raw
device pointer.  There is NO fallback: if the library is missing, importing the compute API raises.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmfm_b200.so")

c_f32p = C.c_void_p
c_u32p = C.c_void_p
c_u8p = C.c_void_p
c_i32p = C.c_void_p


class TargetDesc(C.Structure):
    _fields_ = [
        ("kind", C.c_int), ("dim", C.c_int), ("beta", C.c_float),
        ("n_modes", C.c_int), ("modes", c_f32p), ("stds", c_f32p), ("weights", c_f32p),
        ("phi_a", C.c_float), ("phi_beta", C.c_float),
        ("counts", c_f32p), ("kinv", c_f32p), ("kinv_mu", c_f32p), ("kinv_diag", c_f32p), ("kinv_split", c_f32p),
        ("mu", C.c_float), ("log_norm", C.c_float), ("poisson_a", C.c_float),
        ("chol", c_f32p), ("chol_t", c_f32p), ("chol_sq_t", c_f32p), ("mu_vec", c_f32p),
        ("gauss_mean", C.c_float), ("gauss_std", C.c_float),
    ]


class FieldDesc(C.Structure):
    _fields_ = [
        ("dim", C.c_int), ("hidden", C.c_int), ("fourier_dim", C.c_int),
        ("params", c_f32p), ("w_off", C.c_longlong * 8), ("b_off", C.c_longlong * 8),
        ("n_params", C.c_longlong), ("omega", c_f32p), ("grad_clip", C.c_float),
        ("ref_mean", C.c_float), ("ref_std", C.c_float), ("act", C.c_int),
        ("ref_kind", C.c_int), ("ref_log_norm", C.c_float), ("ref_band", c_f32p),
        ("hidden_t", C.c_int * 2), ("hidden_x", C.c_int * 2), ("hidden_xt", C.c_int * 2),
    ]


class OdeOpts(C.Structure):
    _fields_ = [("rtol", C.c_float), ("atol", C.c_float), ("mxstep", C.c_int), ("hutch", C.c_int),
                ("n_times", C.c_int)]


TARGET_GMM, TARGET_PHI4, TARGET_PINES, TARGET_GAUSS, TARGET_PINES_WHITE = 0, 1, 2, 3, 4
ACTIVATIONS = {"relu": 0, "tanh": 1, "elu": 2, "gelu": 3, "swish": 4}
REF_INDEP_GAUSS, REF_PHI4_BASE = 0, 1
REF_BAND_MAX_DIM = 12192
FLOW_RW_MH, FLOW_INDEP_MH = 0, 1

_PT, _FP, _OP = C.POINTER(TargetDesc), C.POINTER(FieldDesc), C.POINTER(OdeOpts)
_S = C.c_void_p  # stream

# name -> (restype, argtypes); must list every symbol include/mfm_b200.h declares.
SIGNATURES = {
    "mfm_last_error": (C.c_char_p, []),
    "mfm_version": (C.c_int, []),
    "mfm_launch_count": (C.c_ulonglong, []),
    "mfm_set_gemm_backend": (None, [C.c_int]),
    "mfm_set_gemm_raw_hi": (None, [C.c_int]),
    "mfm_set_gemm_cross_bf16": (None, [C.c_int]),
    "mfm_set_gemm_streamk": (None, [C.c_int]),
    "mfm_set_gemm_h16": (None, [C.c_int]),
    "mfm_gemm_describe": (C.c_char_p, []),
    "mfm_gemm_h16_enabled": (C.c_int, []),
    "mfm_absmax": (C.c_int, [c_f32p, C.c_longlong, C.c_int, C.c_int, c_f32p, _S]),
    "mfm_gemm_dense": (C.c_int, [C.c_int, C.c_int, C.c_int, c_f32p, C.c_longlong, c_f32p, C.c_longlong, c_f32p, C.c_int, c_f32p, C.c_longlong,
                                 c_f32p, c_f32p, c_f32p, c_f32p, _S]),
    "mfm_gemm_presplit": (C.c_int, [c_f32p, c_f32p, C.c_longlong, _S]),
    "mfm_gemm_register_mirror": (None, [c_f32p, C.c_longlong, c_f32p]),
    "mfm_debug_gemm_plan": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_int]),
    "mfm_gemm_tf32x3_gated": (C.c_int, [C.c_int, C.c_int, C.c_int, c_f32p, C.c_longlong, c_f32p, C.c_longlong, c_f32p, C.c_longlong,
                                        c_f32p, C.c_longlong, c_f32p, C.c_longlong, _S]),
    "mfm_gemm_tf32x3_rows": (C.c_int, [C.c_int, C.c_int, C.c_int, c_f32p, C.c_longlong, c_f32p, C.c_longlong, c_f32p, c_f32p, C.c_longlong,
                                       C.c_void_p, _S]),
    "mfm_importance_weights": (C.c_int, [c_f32p, c_f32p, c_f32p, C.c_int, c_f32p, c_f32p, _S]),
    "mfm_random_choice_workspace_bytes": (C.c_size_t, [C.c_int]),
    "mfm_random_choice": (C.c_int, [c_u32p, C.c_int, c_f32p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, _S]),
    "mfm_gather_rows": (C.c_int, [c_f32p, C.c_void_p, C.c_int, C.c_int, C.c_int, c_f32p, _S]),
    "mfm_pairwise_workspace_bytes": (C.c_size_t, [C.c_int]),
    "mfm_stein_disc": (C.c_int, [c_f32p, c_f32p, C.c_int, C.c_int, C.c_float, c_f32p, C.c_void_p, C.c_size_t, _S]),
    "mfm_max_mean_disc": (C.c_int, [c_f32p, c_f32p, C.c_int, C.c_int, c_f32p, C.c_void_p, C.c_size_t, _S]),
    "mfm_set_rng_x64": (None, [C.c_int]),
    "mfm_rng_x64_enabled": (C.c_int, []),
    "mfm_threefry_split": (C.c_int, [c_u32p, C.c_int, c_u32p, _S]),
    "mfm_threefry_split_batched": (C.c_int, [c_u32p, C.c_int, C.c_int, c_u32p, _S]),
    "mfm_threefry_bits": (C.c_int, [c_u32p, C.c_longlong, c_u32p, _S]),
    "mfm_threefry_uniform": (C.c_int, [c_u32p, C.c_longlong, C.c_double, C.c_double, c_f32p, _S]),
    "mfm_threefry_normal": (C.c_int, [c_u32p, C.c_longlong, c_f32p, _S]),
    "mfm_threefry_uniform_batched": (C.c_int, [c_u32p, C.c_int, C.c_int, C.c_double, C.c_double, c_f32p, _S]),
    "mfm_threefry_normal_batched": (C.c_int, [c_u32p, C.c_int, C.c_int, c_f32p, _S]),
    "mfm_host_threefry_split": (None, [C.POINTER(C.c_uint32), C.c_int, C.POINTER(C.c_uint32)]),
    "mfm_gemm_tf32x3": (C.c_int, [C.c_int, C.c_int, C.c_int, c_f32p, C.c_longlong, C.c_int, c_f32p, C.c_longlong,
                                  C.c_int, c_f32p, C.c_int, c_f32p, C.c_longlong, _S]),
    "mfm_target_workspace_bytes": (C.c_size_t, [_PT, C.c_int]),
    "mfm_logdensity_and_grad": (C.c_int, [_PT, C.c_int, c_f32p, c_f32p, c_f32p, c_f32p, C.c_void_p, C.c_size_t, _S]),
    "mfm_mala_workspace_bytes": (C.c_size_t, [_PT, C.c_int]),
    "mfm_mala_step": (C.c_int, [_PT, c_u32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, c_f32p, c_f32p, c_f32p,
                                c_f32p, c_u8p, c_f32p, c_f32p, C.c_void_p, C.c_size_t, _S]),
    "mfm_ode_workspace_bytes": (C.c_size_t, [_FP, _PT, _OP, C.c_int]),
    "mfm_ode_flow": (C.c_int, [_FP, _PT, _OP, C.c_int, C.c_int, c_u32p, c_f32p, c_f32p, c_f32p, c_i32p,
                               C.c_void_p, C.c_size_t, _S]),
    "mfm_field_eval": (C.c_int, [_FP, _PT, _OP, C.c_int, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p,
                                 C.c_void_p, C.c_size_t, _S]),
    "mfm_flow_mh_workspace_bytes": (C.c_size_t, [_FP, _PT, _OP, C.c_int]),
    "mfm_flow_mh_step": (C.c_int, [_FP, _PT, _OP, C.c_int, c_u32p, C.c_int, C.c_int, C.c_int, C.c_int, c_f32p, c_f32p, c_f32p,
                                   c_f32p, c_u8p, c_f32p, c_f32p, c_i32p, C.c_void_p, C.c_size_t, _S]),
    "mfm_flow_cis_workspace_bytes": (C.c_size_t, [_FP, _PT, _OP, C.c_int, C.c_int]),
    "mfm_flow_cis_step": (C.c_int, [_FP, _PT, _OP, C.c_int, c_u32p, C.c_int, C.c_int, C.c_int, C.c_int, c_f32p, c_f32p,
                                    c_f32p, c_u8p, c_f32p, c_f32p, c_i32p, C.c_void_p, C.c_size_t, _S]),
    "mfm_ref_sample": (C.c_int, [_FP, c_u32p, C.c_int, c_f32p, _S]),
    "mfm_ref_logprob": (C.c_int, [_FP, C.c_int, c_f32p, c_f32p, _S]),
    "mfm_fm_workspace_bytes": (C.c_size_t, [_FP, _PT, C.c_int]),
    "mfm_fm_loss_grad": (C.c_int, [_FP, _PT, c_u32p, C.c_int, C.c_int, C.c_int, C.c_float, c_f32p, c_f32p, c_f32p,
                                   C.c_void_p, C.c_size_t, _S]),
    "mfm_fm_loss_grad_uncond": (C.c_int, [_FP, _PT, c_u32p, C.c_int, C.c_int, C.c_int, C.c_float, c_f32p, c_f32p, c_f32p,
                                   C.c_void_p, C.c_size_t, _S]),
    "mfm_fm_loss_grad_part": (C.c_int, [_FP, _PT, c_u32p, C.c_int, C.c_int, C.c_int, C.c_float, c_f32p, c_f32p, c_f32p,
                                        C.c_void_p, C.c_size_t, C.c_int, _S]),
    "mfm_fm_loss_grad_from_batch": (C.c_int, [_FP, _PT, C.c_int, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p,
                                              C.c_void_p, C.c_size_t, _S]),
    "mfm_tempering_beta": (C.c_int, [c_f32p, C.c_int, c_f32p, C.c_float, c_f32p, _S]),
    "mfm_adamw_step": (C.c_int, [c_f32p, c_f32p, c_f32p, c_f32p, c_u8p, C.c_longlong, c_i32p, C.c_float, C.c_int, C.c_int,
                                 C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int, _S]),
}

_lib = None


def load():
    """Load the CUDA library.  Raises (never falls back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -m mfm_b200._build` (nvcc, sm_100a). "
            "mfm_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class MfmError(RuntimeError):
    pass


def check(rc: int):
    if rc != 0:
        msg = load().mfm_last_error()
        raise MfmError(f"mfm_b200 error {rc}: {msg.decode() if msg else ''}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "mfm_b200 needs contiguous CUDA tensors"
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


_ws_cache: dict = {}
_ws_generation = 0


def workspace_generation() -> int:
    """Bumped whenever a cached workspace is re-allocated: holders of raw pointers into one (a captured CUDA graph)
    compare it with the value they saw and re-capture."""
    return _ws_generation


def workspace(nbytes: int, device, tag="default"):
    """Grow-only scratch buffer per (device, tag).  Growing REPLACES the tensor; the old one stays alive in
    `_ws_retired` while the generation counter tells graph holders to re-capture (a replay between the two would
    otherwise touch freed memory)."""
    global _ws_generation
    key = (str(device), tag)
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        if buf is not None:
            _ws_retired.append(buf)
            del _ws_retired[:-4]
            _ws_generation += 1
        buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
        _ws_cache[key] = buf
    return buf


_ws_retired: list = []
