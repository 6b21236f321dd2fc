"""ctypes binding of libjimm_b200.so (include/jimm_b200.h).  No CPU fallback: if the CUDA library is missing or no
B200 is present, calls raise."""

from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libjimm_b200.so")

F32, F16, BF16, I32 = 0, 1, 2, 3
PARAM_TRANSPOSED = 1
KIND_VIT, KIND_CLIP, KIND_SIGLIP, KIND_TOWER, KIND_ENCODER, KIND_MAPHEAD = 0, 1, 2, 3, 4, 5
POOL_CLS, POOL_MAP = 0, 1
ACT_GELU_TANH, ACT_QUICK_GELU = 0, 1
TPOOL_EOT_ARGMAX, TPOOL_LAST = 0, 1


class Config(C.Structure):
    """jimm_config_t"""

    _fields_ = [
        ("kind", C.c_int),
        ("img_size", C.c_int), ("patch", C.c_int), ("in_ch", C.c_int), ("v_width", C.c_int), ("v_layers", C.c_int),
        ("v_heads", C.c_int), ("v_mlp", C.c_int),
        ("pooling", C.c_int),
        ("pre_norm", C.c_int), ("patch_bias", C.c_int), ("v_act", C.c_int),
        ("v_eps_outer", C.c_float), ("v_eps_block", C.c_float),
        ("num_classes", C.c_int),
        ("ctx_len", C.c_int), ("vocab", C.c_int), ("t_width", C.c_int), ("t_heads", C.c_int), ("t_layers", C.c_int),
        ("t_mlp", C.c_int),
        ("t_act", C.c_int), ("t_causal", C.c_int), ("t_pool", C.c_int), ("t_head_bias", C.c_int),
        ("t_eps_outer", C.c_float), ("t_eps_block", C.c_float),
        ("compute_dtype", C.c_int),
    ]


_vp, _i, _f, _fp, _ip = C.c_void_p, C.c_int, C.c_float, C.c_void_p, C.c_void_p

# name -> (restype, argtypes): every symbol include/jimm_b200.h declares
class PreprocConfig(C.Structure):
    """jimm_preproc_config_t"""

    _fields_ = [
        ("height", C.c_int), ("width", C.c_int), ("shortest_edge", C.c_int), ("crop_h", C.c_int), ("crop_w", C.c_int),
        ("resample", C.c_int), ("rescale_factor", C.c_double), ("mean", C.c_float * 3), ("std", C.c_float * 3),
    ]


SIGNATURES = {
    "jimm_last_error": (C.c_char_p, []),
    "jimm_abi_version": (_i, []),
    "jimm_launch_count": (C.c_longlong, []),
    "jimm_graph_replay_count": (C.c_longlong, []),
    "jimm_model_create": (_i, [C.POINTER(Config), _i, C.POINTER(_vp)]),
    "jimm_model_set_param": (_i, [_vp, C.c_char_p, _vp, C.POINTER(C.c_int64), _i, _i]),
    "jimm_model_set_param_ref": (_i, [_vp, C.c_char_p, _vp, C.POINTER(C.c_int64), _i, _i, _i]),
    "jimm_model_finalize": (_i, [_vp, _i]),
    "jimm_model_destroy": (_i, [_vp]),
    "jimm_model_output_dim": (_i, [_vp, C.POINTER(_i), C.POINTER(_i)]),
    "jimm_model_max_batch": (_i, [_vp]),
    "jimm_vit_forward": (_i, [_vp, _vp, _i, _i, _fp, _vp]),
    "jimm_encode_image": (_i, [_vp, _vp, _i, _i, _fp, _vp]),
    "jimm_encode_text": (_i, [_vp, _ip, _i, _i, _fp, _vp]),
    "jimm_contrastive_logits": (_i, [_vp, _fp, _i, _fp, _i, _fp, _vp]),
    "jimm_dual_encode": (_i, [_vp, _vp, _i, _i, _ip, _i, _i, _fp, _fp, _vp]),
    "jimm_dual_forward": (_i, [_vp, _vp, _i, _i, _ip, _i, _i, _fp, _vp]),
    "jimm_encoder_forward": (_i, [_vp, _fp, _i, _i, _fp, _vp]),
    "jimm_map_head_forward": (_i, [_vp, _fp, _i, _i, _fp, _vp]),
    "jimm_vit_forward_host": (_i, [_vp, _vp, _i, _i, _fp, _vp]),
    "jimm_dual_forward_host": (_i, [_vp, _vp, _i, _i, _ip, _i, _i, _fp, _vp]),
    "jimm_vit_forward_host_u8": (_i, [_vp, _vp, _vp, _i, _i, _i, _fp, _vp]),
    "jimm_comm_init": (_i, [_vp, _i, _i, _i, C.c_char_p]),
    "jimm_comm_connect": (_i, [_vp, C.c_char_p]),
    "jimm_comm_contrastive_logits": (_i, [_vp, _fp, _fp, _i, _fp, _vp]),
    "jimm_comm_status": (_i, [_vp]),
    "jimm_comm_gathered": (_i, [_vp, C.POINTER(_vp), C.POINTER(_i)]),
    "jimm_profile_begin": (_i, [_vp]),
    "jimm_profile_end": (_i, [_vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_longlong)]),
    "jimm_k_gemm": (_i, [_i, _i, _vp, _i, _vp, _i, _i, _i, _i, _fp, _i, _fp, _fp, _i, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "jimm_k_gemm_ex": (_i, [_i, _vp, _i, _vp, _i, _i, _i, _i, _fp, _i, _fp, _fp, _i, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "jimm_k_layernorm": (_i, [_fp, _i, _i, _i, _ip, _fp, _fp, _f, _vp, _i, _i, _i, _i, _vp]),
    "jimm_k_layernorm_ex": (_i, [_fp, _i, _i, _i, _ip, _fp, _fp, _f, _vp, _i, _i, _i, _i, _i, _vp]),
    "jimm_k_attention": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _i, _vp]),
    "jimm_k_attention_ex": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "jimm_k_map_attention": (_i, [_fp, _vp, _i, _vp, _i, _i, _i, _i, _vp]),
    "jimm_k_patchify": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _i, _vp]),
    "jimm_k_activation": (_i, [_fp, _fp, C.c_longlong, _i, _vp]),
    "jimm_k_embed": (_i, [_ip, _fp, _fp, _fp, _i, _i, _i, _i, _vp]),
    "jimm_k_l2_normalize": (_i, [_fp, _fp, _i, _i, _i, _vp]),
    "jimm_k_logits": (_i, [_fp, _fp, _fp, _fp, _fp, _i, _i, _i, _i, _vp]),
    "jimm_k_l2_probe": (_i, [_vp, _i, _i, _i, _i, C.POINTER(C.c_float), _vp]),
    "jimm_postprocess": (_i, [_fp, _i, _i, _i, _i, _fp, _i, _ip, _ip, _vp]),
    "jimm_preproc_create": (_i, [C.POINTER(PreprocConfig), _i, C.POINTER(_vp)]),
    "jimm_preproc_output_size": (_i, [_vp, _i, _i, C.POINTER(_i), C.POINTER(_i)]),
    "jimm_preproc_run": (_i, [_vp, _vp, _i, _i, _i, _vp, _i, _vp]),
    "jimm_preproc_destroy": (_i, [_vp]),
    "jimm_k_resample_coeffs": (_i, [_i, _i, _i, C.POINTER(_i), _ip, _ip, _ip, _i]),
}

_lib = None


class JimmError(RuntimeError):
    pass


def load():
    """Load the shared library (building nothing: run `python -m jimm_b200.build` / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise JimmError(f"{LIB_PATH} not found: build it with `python -m jimm_b200.build` (there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    return load().jimm_last_error().decode("utf-8", "replace")


def check(rc: int):
    """Map a negative status to the exception type the reference would raise (ValueError for bad arguments /
    shapes, AssertionError is reserved for loader checks done in Python)."""
    if rc == 0:
        return
    msg = last_error()
    if rc == -1:
        raise ValueError(msg)
    raise JimmError(f"jimm_b200 error {rc}: {msg}")
