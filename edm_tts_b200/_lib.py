"""ctypes binding of libedm_s2a.so (the C ABI declared in include/edm_s2a.h).

There is no fallback: if the shared library is missing or a call fails, an exception is raised. PyTorch is only used by
callers for device memory and streams; every argument crossing this boundary is a raw pointer or a scalar.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libedm_s2a.so")

EPI_BF16, EPI_SWISH_BF16, EPI_QKV_ROPE, EPI_RESID_F32, EPI_F32, EPI_GLU_BF16 = range(6)
EPI_ARGMAX = 10
EPI_GELU_BF16 = 11


class S2AConfig(C.Structure):
    _fields_ = [
        ("hidden", C.c_int), ("heads", C.c_int), ("depth", C.c_int), ("ff_mult", C.c_int), ("conv_kernel", C.c_int),
        ("num_quantizers", C.c_int), ("num_codes", C.c_int), ("num_semantic", C.c_int), ("n_injection", C.c_int),
        ("injection_layers", C.c_int * 4), ("residual", C.c_int), ("max_positions", C.c_int),
    ]


class T2SConfig(C.Structure):
    _fields_ = [
        ("hidden", C.c_int), ("heads", C.c_int), ("depth", C.c_int), ("lp_heads", C.c_int), ("lp_depth", C.c_int), ("ff_mult", C.c_int),
        ("conv_kernel", C.c_int), ("text_vocab", C.c_int), ("semantic_vocab", C.c_int), ("num_special", C.c_int), ("max_positions", C.c_int),
    ]


class EdmError(RuntimeError):
    pass


_lib = None

_vp, _i, _ll, _f, _u, _ull, _sz = C.c_void_p, C.c_int, C.c_longlong, C.c_float, C.c_uint, C.c_ulonglong, C.c_size_t

_SIGNATURES = {
    "edm_abi_version": (_i, []),
    "edm_last_error": (C.c_char_p, []),
    "edm_launch_count": (_ull, []),
    "edm_prof_enable": (None, [_i]),
    "edm_prof_collect": (_i, [C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "edm_gemm_bf16": (_i, [_vp, _ll, _vp, _ll, _i, _i, _i, _i, _vp, _vp, _ll, _f, _vp, _vp, _i, _i, _vp]),
    "edm_attention": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "edm_attention_varlen": (_i, [_vp, _i, _vp, _i, _vp, _vp]),
    "edm_layernorm": (_i, [_vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _vp]),
    "edm_gemm_resid_layernorm": (_i, [_vp, _ll, _vp, _ll, _i, _i, _vp, _vp, _f, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _vp, _i, _vp]),
    "edm_conv_module": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _i, _i, _vp]),
    "edm_conv_module_varlen": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp]),
    "edm_sample": (_i, [_vp, _ll, _i, _vp, _i, _ull, _u, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "edm_remask": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _f, _f, _ull, _u, _vp]),
    "edm_rvq_encode_tc": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "edm_kmeans_assign": (_i, [_vp, _ll, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "edm_kmeans_update_workspace_bytes": (_sz, [_ll, _i, _i]),
    "edm_kmeans_update": (_i, [_vp, _ll, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "edm_dac_conv": (_i, [_vp, _ll, _i, _ll, _i, _vp, _i, _i, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _ll, _vp, _ll, _i, _i, _vp, _i, _vp]),
    "edm_dac_conv_last": (_i, [_vp, _ll, _i, _i, _i, _vp, C.c_float, _vp, _i, _vp]),
    "edm_dac_resunit": (_i, [_vp, _ll, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _vp, _ll, _i, _i, _vp]),
    "edm_dac_conv_first": (_i, [_vp, _i, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "edm_dac_zero_rows": (_i, [_vp, _ll, _vp, _i, _i, _vp]),
    "edm_hubert_conv0": (_i, [_vp, _ll, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "edm_hubert_ln512": (_i, [_vp, _vp, _i, _vp, _vp, _i, _vp, _vp]),
    "edm_hubert_pad_rows": (_i, [_vp, _vp, _i, _vp, _vp]),
    "edm_hubert_pos_conv": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "edm_codes_to_features": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "edm_s2a_num_weights": (_i, [C.POINTER(S2AConfig)]),
    "edm_s2a_weight_name": (C.c_char_p, [C.POINTER(S2AConfig), _i]),
    "edm_s2a_create": (_vp, [C.POINTER(S2AConfig), C.POINTER(_vp), _i]),
    "edm_s2a_destroy": (None, [_vp]),
    "edm_s2a_workspace_bytes": (_sz, [_vp, _i, _i, _i]),
    "edm_s2a_bind": (_i, [_vp, _vp, _sz, _i, _i, _i]),
    "edm_s2a_workspace_bytes_varlen": (_sz, [_vp, _i, _vp, _vp]),
    "edm_s2a_bind_varlen": (_i, [_vp, _vp, _sz, _i, _vp, _vp, _vp]),
    "edm_s2a_bind_masked": (_i, [_vp, _vp, _sz, _i, _vp, _vp, _vp]),
    "edm_s2a_buffer": (_vp, [_vp, C.c_char_p, C.POINTER(_sz)]),
    "edm_s2a_set_batch_offset": (_i, [_vp, _ll]),
    "edm_s2a_set_seed_buffer": (_i, [_vp, _vp]),
    "edm_s2a_set_keep_logits": (_i, [_vp, _i]),
    "edm_s2a_set_low_latency": (_i, [_vp, _i]),
    "edm_s2a_set_prompt_injections": (_i, [_vp, _vp]),
    "edm_s2a_build_input": (_i, [_vp, _vp, _vp, _vp, _i, _vp]),
    "edm_s2a_first_level": (_i, [_vp, _vp, _vp]),
    "edm_s2a_step": (_i, [_vp, _i, _i, _f, _ull, _vp, _vp, _vp, _vp, _vp]),
    "edm_s2a_full_pass": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "edm_s2a_decode": (_i, [_vp, _vp, _vp, _vp, _i, _i, _f, _ull, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "edm_t2s_num_weights": (_i, [C.POINTER(T2SConfig)]),
    "edm_t2s_weight_name": (C.c_char_p, [C.POINTER(T2SConfig), _i]),
    "edm_t2s_create": (_vp, [C.POINTER(T2SConfig), C.POINTER(_vp), _i]),
    "edm_t2s_destroy": (None, [_vp]),
    "edm_t2s_workspace_bytes": (_sz, [_vp, _i]),
    "edm_t2s_bind": (_i, [_vp, _vp, _sz, _i]),
    "edm_t2s_workspace_bytes_batch": (_sz, [_vp, _i, _i]),
    "edm_t2s_bind_batch": (_i, [_vp, _vp, _sz, _i, _i]),
    "edm_t2s_set_low_latency": (_i, [_vp, _i]),
    "edm_t2s_set_batch_offset": (_i, [_vp, _ll]),
    "edm_t2s_buffer": (_vp, [_vp, C.c_char_p, C.POINTER(_sz)]),
    "edm_t2s_predict_length": (_i, [_vp, _vp, _i, _vp, _vp]),
    "edm_t2s_predict_length_batch": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "edm_t2s_begin": (_i, [_vp, _vp, _i, _i, _vp]),
    "edm_t2s_begin_batch": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "edm_t2s_logits": (_i, [_vp, _vp, _vp]),
    "edm_t2s_step": (_i, [_vp, _i, _i, _f, _ull, _vp, _vp, _vp, _vp, _vp]),
    "edm_t2s_result": (_i, [_vp, _vp, _vp]),
    "edm_t2s_decode": (_i, [_vp, _vp, _i, _i, _i, _f, _ull, _vp, _vp, _vp, _vp, _vp, _vp]),
    "edm_t2s_decode_batch": (_i, [_vp, _i, _vp, _vp, _vp, _i, _f, _ull, _vp, _vp, _vp, _vp, _vp, _vp]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def lib() -> C.CDLL:
    """Load the extension once; fail loudly when it has not been built (python -c 'import __graft_entry__ as g; g.build()')."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise EdmError(f"{LIB_PATH} not found: build it with __graft_entry__.build(); there is no CPU fallback")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        if handle.edm_abi_version() != 1:
            raise EdmError("libedm_s2a.so ABI version mismatch")
        _lib = handle
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().edm_last_error().decode("utf-8", "replace")
        raise (ValueError if rc == -1 else EdmError)(f"{what or 'edm call'} failed ({rc}): {msg}")


def ptr(t) -> int | None:
    """Device pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "edm ABI takes contiguous CUDA tensors"
    return t.data_ptr()


def stream_ptr() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream
