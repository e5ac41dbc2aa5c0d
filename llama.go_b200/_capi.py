"""ctypes binding of include/llamab200.h.  Loads the in-tree libllamab200.so and fails loudly
when it is missing or cannot drive a GPU: there is no CPU fallback anywhere in this package."""
from __future__ import annotations

import ctypes as C
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libllamab200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "llamab200.h")

_f32p = C.POINTER(C.c_float)
_u32p = C.POINTER(C.c_uint32)
_vp = C.c_void_p


class HParamsC(C.Structure):
    _fields_ = [("vocab", C.c_uint32), ("dim", C.c_uint32), ("mult", C.c_uint32),
                ("heads", C.c_uint32), ("layers", C.c_uint32)]


class LlamaB200Error(RuntimeError):
    pass


_SIGS = {
    "lb_last_error": (C.c_char_p, []),
    "lb_device_count": (C.c_int, []),
    "lb_version": (C.c_char_p, []),
    "lb_kernel_launches": (C.c_uint64, []),
    "lb_model_create": (_vp, [C.POINTER(HParamsC), C.c_int, C.c_uint32, C.c_uint32, C.c_int]),
    "lb_model_free": (None, [_vp]),
    "lb_model_load_ggjt": (_vp, [C.c_char_p, C.c_int, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(HParamsC)]),
    "lb_model_set_tensor": (C.c_int, [_vp, C.c_char_p, C.c_int, _vp, C.c_size_t]),
    "lb_model_get_tensor": (C.c_int, [_vp, C.c_char_p, _f32p, C.c_size_t]),
    "lb_model_init_random": (C.c_int, [_vp, C.c_uint64]),
    "lb_model_weight_bytes": (C.c_uint64, [_vp]),
    "lb_synth_fill_host": (C.c_int, [_f32p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_float, C.c_double]),
    "lb_bench_kernel": (C.c_int, [_vp, C.c_int, C.c_uint32, C.c_uint32, _f32p, C.POINTER(C.c_uint64)]),
    "lb_context_create": (_vp, [_vp, C.c_uint32]),
    "lb_context_free": (None, [_vp]),
    "lb_eval": (C.c_int, [_vp, _u32p, C.c_uint32, C.c_uint32, _f32p]),
    "lb_eval_all_logits": (C.c_int, [_vp, _u32p, C.c_uint32, C.c_uint32, _f32p]),
    "lb_eval_graph": (C.c_int, [_vp, _u32p, C.c_uint32, C.c_uint32, _f32p]),
    "lb_decode_resident": (C.c_int, [_vp, _u32p, C.c_uint32, C.c_uint32, _f32p]),
    "lb_generate_greedy": (C.c_int, [_vp, _u32p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, _u32p]),
    "lb_sample_top_p_top_k": (C.c_int, [_vp, _u32p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.c_uint64, _u32p, _f32p,
                                        _u32p, _u32p]),
    "lb_generate": (C.c_int, [_vp, _u32p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.c_uint32, C.c_uint32,
                              C.c_uint64, _u32p]),
    "lb_context_swap": (C.c_int64, [C.c_uint32, C.c_uint32, _u32p, C.c_uint32, _u32p, _u32p, C.c_uint32, _u32p, C.c_uint32]),
    "lb_context_read_logits": (C.c_int, [_vp, _f32p]),
    "lb_context_read_kv": (C.c_int, [_vp, C.c_uint32, C.c_uint32, C.c_uint32, _f32p, _f32p]),
    "lb_context_read_hidden": (C.c_int, [_vp, C.c_uint32, _f32p]),
    "lb_context_synchronize": (C.c_int, [_vp]),
    "lb_context_mega_trace": (C.c_int, [_vp, C.POINTER(C.c_uint64), C.c_uint32]),
    "lb_eval_stage": (C.c_int, [_vp, _u32p, C.c_uint32, C.c_uint32, _vp, _vp, _f32p]),
    "lb_context_hidden_buffer": (_vp, [_vp]),
    "lb_context_stream": (_vp, [_vp]),
    "lb_context_decode_path": (C.c_char_p, [_vp]),
    "lb_layout_query": (C.c_int, [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32)]),
    "lb_vocab_create": (_vp, [C.c_uint32]),
    "lb_vocab_free": (None, [_vp]),
    "lb_vocab_set": (C.c_int, [_vp, C.c_uint32, C.c_char_p, C.c_uint32, C.c_float]),
    "lb_tokenize": (C.c_int64, [_vp, C.c_char_p, C.c_uint32, C.c_int, _u32p, C.c_uint32]),
    "lb_batch_create": (_vp, [C.POINTER(_vp), C.c_uint32]),
    "lb_batch_free": (None, [_vp]),
    "lb_batch_eval": (C.c_int, [_vp, _u32p, _u32p, _f32p]),
    "lb_batch_decode_resident": (C.c_int, [_vp, _u32p, C.c_uint32, _u32p, _f32p]),
    "lb_batch_read_logits": (C.c_int, [_vp, _f32p]),
    "lb_batch_mega_trace": (C.c_int, [_vp, C.POINTER(C.c_uint64), C.c_uint32]),
    "lb_batch_sample": (C.c_int, [_vp, _u32p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_uint64), _u32p,
                                  _f32p, _u32p, _u32p]),
    "lb_batch_generate": (C.c_int, [_vp, _u32p, _u32p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.c_uint32, C.c_uint32,
                                    C.POINTER(C.c_uint64), _u32p, _f32p]),
    "lb_comm_unique_id": (C.c_int, [_vp]),
    "lb_comm_init": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int]),
    "lb_comm_destroy": (None, []),
    "lb_nccl_version": (C.c_int, []),
    "lb_pipeline_decode": (C.c_int, [C.POINTER(_vp), C.c_uint32, _u32p, C.c_uint32, C.c_uint32, _f32p]),
    "lb_pipeline_prefill": (C.c_int, [C.POINTER(_vp), C.c_uint32, _u32p, C.c_uint32, C.c_uint32]),
    "lb_pipeline_p2p_export": (C.c_int, [C.POINTER(_vp), C.c_uint32, _vp]),
    "lb_pipeline_p2p_import": (C.c_int, [C.POINTER(_vp), C.c_uint32, C.c_char_p, C.c_char_p]),
    "lb_pipeline_p2p_disable": (C.c_int, [C.POINTER(_vp), C.c_uint32]),
    "lb_ml_new_context": (_vp, [C.c_int]),
    "lb_ml_release_context": (None, [_vp]),
    "lb_new_tensor": (_vp, [_vp, C.c_int] + [C.c_uint32] * 5 + [_f32p]),
    "lb_tensor_write": (C.c_int, [_vp, _f32p, C.c_size_t]),
    "lb_tensor_read": (C.c_int, [_vp, _f32p, C.c_size_t]),
    "lb_tensor_shape": (C.c_int, [_vp, C.c_uint32 * 4, C.c_uint32 * 4]),
    "lb_get_rows": (_vp, [_vp, _vp, _vp]),
    "lb_rms_norm": (_vp, [_vp, _vp]),
    "lb_repeat": (_vp, [_vp, _vp, _vp]),
    "lb_mul": (_vp, [_vp, _vp, _vp]),
    "lb_add": (_vp, [_vp, _vp, _vp]),
    "lb_mul_mat": (_vp, [_vp, _vp, _vp]),
    "lb_view_1d": (_vp, [_vp, _vp, C.c_uint32, C.c_uint32]),
    "lb_cpy": (_vp, [_vp, _vp, _vp]),
    "lb_rope": (_vp, [_vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32]),
    "lb_permute": (_vp, [_vp, _vp] + [C.c_uint32] * 4),
    "lb_transpose": (_vp, [_vp, _vp]),
    "lb_reshape_3d": (_vp, [_vp, _vp] + [C.c_uint32] * 3),
    "lb_new_f32": (_vp, [_vp, C.c_float]),
    "lb_scale": (_vp, [_vp, _vp, _vp]),
    "lb_diag_mask_inf": (_vp, [_vp, _vp, C.c_uint32]),
    "lb_soft_max": (_vp, [_vp, _vp]),
    "lb_silu": (_vp, [_vp, _vp]),
    "lb_graph_new": (_vp, []),
    "lb_graph_free": (None, [_vp]),
    "lb_build_forward_expand": (C.c_int, [_vp, _vp]),
    "lb_graph_compute": (C.c_int, [_vp, _vp]),
    "lb_graph_nodes": (C.c_uint32, [_vp]),
}

_lib = None


def header_symbols():
    """Every LB_API symbol include/llamab200.h declares."""
    with open(HEADER_PATH) as f:
        src = f.read()
    return sorted(set(re.findall(r"LB_API[^;]*?\b(lb_[a-z0-9_]+)\s*\(", src, re.S)))


def lib():
    """The loaded C-ABI library (loads on first use; raises if the extension is missing)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LlamaB200Error(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C llama.go_b200/csrc`). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)  # AttributeError if the library does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def last_error() -> str:
    return (lib().lb_last_error() or b"").decode("utf-8", "replace")


def check(rc: int) -> None:
    if rc != 0:
        raise LlamaB200Error(last_error())


def check_ptr(p):
    if not p:
        raise LlamaB200Error(last_error())
    return p


def require_gpu() -> int:
    n = lib().lb_device_count()
    if n <= 0:
        raise LlamaB200Error("no sm_100 (B200) device is visible; this engine has no CPU fallback")
    return n
