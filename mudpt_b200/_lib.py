"""ctypes binding of libmudpt_b200.so (include/mudpt_b200.h).

The product path has no CPU or PyTorch fallback: if the library is missing, or a compute entry
point is called without a Blackwell GPU, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

from . import build as _build

_lib: Optional[C.CDLL] = None
_lib_path: Optional[str] = None

c_f32p = C.c_void_p  # raw device pointers (tensor.data_ptr())

# name -> (restype, argtypes); must list every symbol include/mudpt_b200.h declares
SIGNATURES = {
    "mudpt_abi_version": (C.c_int, []),
    "mudpt_global_last_error": (C.c_char_p, []),
    "mudpt_create": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "mudpt_destroy": (None, [C.c_void_p]),
    "mudpt_last_error": (C.c_char_p, [C.c_void_p]),
    "mudpt_set_weight": (C.c_int, [C.c_void_p, C.c_char_p, c_f32p, C.c_int64, C.c_void_p]),
    "mudpt_weights_complete": (C.c_int, [C.c_void_p]),
    "mudpt_vision_forward": (C.c_int, [C.c_void_p, c_f32p, C.c_int32, c_f32p, c_f32p, C.c_void_p]),
    "mudpt_vision_backward": (C.c_int, [C.c_void_p, c_f32p, c_f32p, C.c_void_p]),
    "mudpt_vision_backward_images": (C.c_int, [C.c_void_p, c_f32p, c_f32p, c_f32p, C.c_void_p]),
    "mudpt_vision_pgd_step": (C.c_int, [C.c_void_p, c_f32p, c_f32p, c_f32p, c_f32p, C.c_void_p, C.c_void_p, C.c_float,
                                         C.c_float, C.c_void_p]),
    "mudpt_text_set_classes": (C.c_int, [C.c_void_p, c_f32p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "mudpt_text_set_classes_ragged": (C.c_int, [C.c_void_p, c_f32p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mudpt_text_forward": (C.c_int, [C.c_void_p, c_f32p, C.c_int32, c_f32p, C.c_void_p]),
    "mudpt_text_backward": (C.c_int, [C.c_void_p, c_f32p, c_f32p, c_f32p, C.c_void_p]),
    "mudpt_vision_infer": (C.c_int, [C.c_void_p, c_f32p, C.c_int32, c_f32p, c_f32p, C.c_void_p]),
    "mudpt_text_infer": (C.c_int, [C.c_void_p, c_f32p, C.c_int32, c_f32p, C.c_void_p]),
    "mudpt_workspace_bytes": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_int64)]),
    "mudpt_logits_head": (C.c_int, [C.c_void_p, c_f32p, c_f32p, C.c_void_p, C.c_int32, C.c_int32, C.c_float,
                                    c_f32p, c_f32p, c_f32p, c_f32p, C.c_void_p]),
    "mudpt_logits_backward": (C.c_int, [C.c_void_p, c_f32p, c_f32p, c_f32p, C.c_int32, C.c_int32, c_f32p, c_f32p, C.c_void_p]),
    "mudpt_layernorm_forward": (C.c_int, [c_f32p, c_f32p, c_f32p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "mudpt_layernorm_backward": (C.c_int, [c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "mudpt_layernorm_backward_stream": (C.c_int, [C.c_void_p, C.c_void_p, c_f32p, c_f32p, C.c_void_p, C.c_int32, c_f32p, C.c_void_p,
                                                  C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "mudpt_splice_forward": (C.c_int, [c_f32p, c_f32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "mudpt_splice_backward": (C.c_int, [c_f32p, C.c_void_p, c_f32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                        C.c_int32, C.c_void_p]),
    "mudpt_attention_forward": (C.c_int, [C.c_void_p, C.c_void_p, c_f32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "mudpt_attention_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, c_f32p, c_f32p, C.c_void_p, C.c_int32,
                                           C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "mudpt_attention_varlen_forward": (C.c_int, [C.c_void_p, C.c_void_p, c_f32p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                                 C.c_void_p]),
    "mudpt_attention_varlen_backward": (C.c_int, [C.c_void_p, C.c_void_p, c_f32p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                                  C.c_int32, C.c_void_p]),
    "mudpt_gemm_bf16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                  C.c_void_p, c_f32p, c_f32p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "mudpt_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int32]),
    "mudpt_gemm_fused": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "mudpt_gemm_dots_span": (C.c_int32, [C.c_int32]),
    "mudpt_rowstats": (C.c_int, [c_f32p, C.c_void_p, c_f32p, C.c_int32, C.c_int32, C.c_void_p]),
    "mudpt_fold_layernorm": (C.c_int, [c_f32p, c_f32p, c_f32p, c_f32p, C.c_void_p, C.c_void_p, c_f32p, c_f32p, c_f32p,
                                       C.c_int32, C.c_int32, C.c_void_p]),
    "mudpt_attention_backward_dots": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, c_f32p, c_f32p, C.c_void_p, C.c_int32,
                                                C.c_int32, C.c_int32, C.c_int32, c_f32p, c_f32p, C.c_void_p]),
    "mudpt_set_attention_tc": (C.c_int, [C.c_int32]),
    "mudpt_im2col": (C.c_int, [c_f32p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "mudpt_col2im": (C.c_int, [c_f32p, c_f32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "mudpt_pgd_linf_update": (C.c_int, [c_f32p, C.c_int32, c_f32p, c_f32p, c_f32p, C.c_int32, C.c_int32, C.c_int32,
                                         C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_void_p]),
    "mudpt_cast_bf16": (C.c_int, [c_f32p, C.c_void_p, C.c_int64, C.c_void_p]),
    "mudpt_prompt_forward": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mudpt_prompt_backward": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mudpt_sgd_step": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_int64),
                                 C.c_int32, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int32, C.c_int32, C.c_void_p]),
    "mudpt_augment_workspace_bytes": (C.c_int64, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32]),
    "mudpt_augment_images": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_float),
                                       C.POINTER(C.c_float), C.c_void_p, C.c_int64, c_f32p, C.c_void_p]),
    "mudpt_debug_buffer": (C.c_int, [C.c_void_p, C.c_int32, C.c_char_p, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "mudpt_profile_begin": (C.c_int, [C.c_void_p]),
    "mudpt_peer_all_gather_rows": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "mudpt_peer_reduce_scatter_rows": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "mudpt_profile_end": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.c_int32]),
    "mudpt_profile_end_bound": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.c_int32, C.c_double, C.c_double]),
    "mudpt_launch_count": (C.c_int64, [C.c_void_p]),
}


class Config(C.Structure):
    """mudpt_config (include/mudpt_b200.h)."""
    _fields_ = [(n, C.c_int32) for n in (
        "embed_dim", "image_resolution", "vision_layers", "vision_width", "vision_patch_size",
        "context_length", "transformer_width", "transformer_heads", "transformer_layers",
        "n_ctx", "prompt_depth", "device")]


class GemmEpilogue(C.Structure):
    """mudpt_gemm_epilogue (include/mudpt_b200.h): every epilogue of the tcgen05 GEMM, for tests and profiling."""
    _fields_ = [("mode", C.c_int32), ("ldc", C.c_int32), ("out0", C.c_void_p), ("out1", C.c_void_p), ("out2", C.c_void_p),
                ("bias", C.c_void_p), ("resid", C.c_void_p), ("aux", C.c_void_p), ("ln_stats", C.c_void_p),
                ("ln_parts", C.c_int32), ("ln_width", C.c_int32), ("ln_eps", C.c_float), ("dot_parts", C.c_int32),
                ("colsum", C.c_void_p), ("stats_out", C.c_void_p), ("splice_prompt", C.c_void_p),
                ("splice_row0", C.c_int32), ("splice_n", C.c_int32), ("splice_L", C.c_int32), ("stream_k", C.c_int32),
                ("x2", C.c_void_p), ("dots", C.c_void_p), ("sb", C.c_void_p), ("dots_out", C.c_void_p)]


class PromptArgs(C.Structure):
    """mudpt_prompt_args (include/mudpt_b200.h)."""
    _fields_ = ([(k, C.c_int32) for k in ("n", "depth", "dt", "dv")] + [("eps", C.c_float)] +
                [(k, C.c_void_p) for k in ("ctx", "deep", "We", "be", "Wd", "bd", "vctx", "vdeep", "Wv", "bv", "ln_g", "ln_b", "pos",
                                           "P_v", "P_t", "ln_in", "dP_v", "dP_t", "u", "d_ctx", "d_deep", "d_We", "d_be", "d_Wd",
                                           "d_bd", "d_vctx", "d_vdeep", "d_Wv", "d_bv")])


def library_path() -> str:
    bringup = os.environ.get("MUDPT_BRINGUP_LIB", "0") == "1"
    return _build.lib_path(bringup)


def load() -> C.CDLL:
    global _lib, _lib_path
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise RuntimeError(
            f"mudpt_b200: native library {path} not found. Build it with `python -m mudpt_b200.build` "
            "(or __graft_entry__.build()). There is no CPU / PyTorch fallback for the hot path.")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    if lib.mudpt_abi_version() != 1:
        raise RuntimeError("mudpt_b200: ABI version mismatch between _lib.py and the shared library")
    if os.environ.get("MUDPT_BRINGUP_LIB", "0") == "1" and os.environ.get("MUDPT_BRINGUP_SIMT_GEMM", "0") == "1":
        import sys
        sys.stderr.write("mudpt_b200: BRING-UP DIAGNOSTIC: SIMT GEMM enabled (not the product path)\n")
        lib.mudpt_bringup_simt_gemm.restype = C.c_int
        lib.mudpt_bringup_simt_gemm.argtypes = [C.c_int]
        lib.mudpt_bringup_simt_gemm(1)
    _lib, _lib_path = lib, path
    return lib


def stream_ptr(device=None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "mudpt_b200: tensors crossing the C ABI must be contiguous CUDA tensors"
    return t.data_ptr()


def check(rc: int, handle=None) -> None:
    if rc < 0:
        lib = load()
        msg = lib.mudpt_last_error(handle) if handle else lib.mudpt_global_last_error()
        raise RuntimeError("mudpt_b200: " + (msg.decode() if msg else "unknown error"))
