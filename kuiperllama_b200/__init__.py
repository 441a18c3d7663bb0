"""kuiperllama_b200 -- B200-native (sm_100a) single-batch decoder behind KuiperLLama's API.

The product is native code:
  * ``lib/libkllm_b200.so``  hand-written CUDA kernels + the C-ABI of ``include/kllm_b200.h``;
  * ``kuiper/``              the C++ host side mirroring the reference's ``kuiper::`` API
                             (base / tensor / op registry / model), built by CMake.
This Python package is only the loader used by tests and ``bench.py``: it dlopens the C-ABI
with ctypes and FAILS LOUDLY when the library is missing or cannot be loaded -- there is no
Python/CPU fallback for any op.
"""
from __future__ import annotations

import ctypes
import ctypes.util
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_int8, c_uint64, c_void_p
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "lib" / "libkllm_b200.so"
HEADER_PATH = PKG_DIR.parent / "include" / "kllm_b200.h"

FLAVOUR_LLAMA2, FLAVOUR_LLAMA3, FLAVOUR_QWEN2 = 0, 1, 2
FLAVOURS = {"llama2": FLAVOUR_LLAMA2, "llama3": FLAVOUR_LLAMA3, "qwen2": FLAVOUR_QWEN2}


class KllmError(RuntimeError):
    pass


class GemvSeg(ctypes.Structure):
    _fields_ = [("w", c_void_p), ("scales", c_void_p), ("bias", c_void_p), ("out", c_void_p),
                ("rows", c_int)]


class GemvJob(ctypes.Structure):
    _fields_ = [("x", c_void_p), ("norm_w", c_void_p), ("norm_eps", c_float),
                ("norm_out", c_void_p), ("in_dim", c_int), ("group_size", c_int),
                ("n_seg", c_int), ("seg", GemvSeg * 3), ("residual", c_void_p),
                ("swiglu_pair", c_int)]


ALLREDUCE_FN = ctypes.CFUNCTYPE(c_int, c_void_p, c_void_p, c_int, c_void_p)


class DecoderDesc(ctypes.Structure):
    _fields_ = [
        ("dim", c_int32), ("hidden_dim", c_int32), ("layer_num", c_int32), ("head_num", c_int32),
        ("kv_head_num", c_int32), ("vocab_size", c_int32), ("seq_len", c_int32),
        ("flavour", c_int32), ("group_size", c_int32),
        ("tok_emb", c_void_p), ("attn_norm", POINTER(c_void_p)), ("ffn_norm", POINTER(c_void_p)),
        ("final_norm", c_void_p),
        ("wq", POINTER(c_void_p)), ("wk", POINTER(c_void_p)), ("wv", POINTER(c_void_p)),
        ("wo", POINTER(c_void_p)), ("w1", POINTER(c_void_p)), ("w2", POINTER(c_void_p)),
        ("w3", POINTER(c_void_p)), ("wcls", c_void_p),
        ("sq", POINTER(c_void_p)), ("sk", POINTER(c_void_p)), ("sv", POINTER(c_void_p)),
        ("so", POINTER(c_void_p)), ("s1", POINTER(c_void_p)), ("s2", POINTER(c_void_p)),
        ("s3", POINTER(c_void_p)), ("scls", c_void_p),
        ("bq", POINTER(c_void_p)), ("bk", POINTER(c_void_p)), ("bv", POINTER(c_void_p)),
        ("tp_size", c_int32), ("tp_rank", c_int32),
        ("allreduce", ALLREDUCE_FN), ("allreduce_ctx", c_void_p), ("comm", c_void_p),
        ("numerics", c_int32),
    ]


# name -> (restype, argtypes); must list EVERY function include/kllm_b200.h declares
# (tests/test_abi.py cross-checks this table against the header and the built library).
_SIGNATURES = {
    "kllm_version": (c_char_p, []),
    "kllm_error_string": (c_char_p, [c_int]),
    "kllm_launch_count": (c_uint64, []),
    "kllm_gemv_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "kllm_gemv_w8": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "kllm_rmsnorm_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_float, c_void_p]),
    "kllm_add_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "kllm_swiglu_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "kllm_sincos_init": (c_int, [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "kllm_rope_f32": (c_int, [c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p,
                              c_void_p, c_void_p]),
    "kllm_mha_decode_f32": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "kllm_embedding_f32": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "kllm_argmax_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "kllm_argmax_f32_sync": (c_int64, [c_void_p, c_int64, c_void_p]),
    "kllm_gemv_fused": (c_int, [POINTER(GemvJob), c_void_p]),
    "kllm_gemm_tf32": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "kllm_gemm_w8": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "kllm_comm_unique_id": (c_int, [c_void_p]),
    "kllm_comm_create": (c_int, [c_int, c_int, c_int, c_int, c_void_p, POINTER(c_void_p)]),
    "kllm_comm_ipc_handle": (c_int, [c_void_p, c_void_p]),
    "kllm_comm_connect": (c_int, [c_void_p, c_void_p]),
    "kllm_comm_allreduce_residual": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "kllm_comm_allreduce": (c_int, [c_void_p, c_void_p, c_int, c_void_p]),
    "kllm_comm_info": (c_int, [c_void_p, POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "kllm_comm_destroy": (None, [c_void_p]),
    "kllm_decoder_create": (c_int, [POINTER(DecoderDesc), c_void_p, POINTER(c_void_p)]),
    "kllm_decoder_destroy": (None, [c_void_p]),
    "kllm_decoder_step": (c_int, [c_void_p, c_int32, c_int32, c_int, POINTER(c_int32)]),
    "kllm_decoder_prompt": (c_int, [c_void_p, POINTER(c_int32), c_int32, c_int32, POINTER(c_int32)]),
    "kllm_decoder_prefill_tf32": (c_int, [c_void_p, POINTER(c_int32), c_int32, c_int32, POINTER(c_int32)]),
    "kllm_decoder_prefill_w8": (c_int, [c_void_p, POINTER(c_int32), c_int32, c_int32, POINTER(c_int32)]),
    "kllm_decoder_generate": (c_int, [c_void_p, c_int32, c_int32, c_int32, POINTER(c_int32),
                                      POINTER(c_int32)]),
    "kllm_decoder_logits": (c_int, [c_void_p, c_void_p]),
    "kllm_decoder_logits_device": (c_void_p, [c_void_p]),
    "kllm_decoder_read_kv": (c_int, [c_void_p, c_void_p, c_void_p]),
    "kllm_decoder_launches_per_step": (c_int, [c_void_p]),
    "kllm_decoder_classifier_rows": (c_int, [c_void_p]),
    "kllm_decoder_engine": (c_char_p, [c_void_p]),
    "kllm_decoder_profile": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int32,
                                     POINTER(c_int32), POINTER(c_int32)]),
}

_lib = None


def load_library(path: str | Path | None = None) -> ctypes.CDLL:
    """dlopen libkllm_b200.so and attach prototypes.  Raises KllmError if it is not there."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    import os
    if path is None and os.environ.get("KLLM_LIB"):  # experiments: a variant build of the same C-ABI
        path = os.environ["KLLM_LIB"]
    p = Path(path) if path else LIB_PATH
    if not p.exists():
        raise KllmError(
            f"{p} is missing: build it with `python -m kuiperllama_b200.build` "
            "(there is no CPU or PyTorch fallback for the decode path)")
    try:
        lib = ctypes.CDLL(str(p))
    except OSError as e:  # pragma: no cover - depends on the host
        raise KllmError(f"cannot load {p}: {e}") from e
    for name, (restype, argtypes) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError = missing export: fail loudly
        fn.restype = restype
        fn.argtypes = argtypes
    if path is None or os.environ.get("KLLM_LIB") == str(path):
        _lib = lib
    return lib


def check(rc: int, what: str = "kllm call") -> None:
    if rc != 0:
        lib = load_library()
        raise KllmError(f"{what} failed: {rc} ({lib.kllm_error_string(rc).decode()})")


from .decoder import Decoder, ModelShape, SHAPES, synth_weights  # noqa: E402

__all__ = ["load_library", "check", "KllmError", "GemvJob", "GemvSeg", "DecoderDesc", "Decoder",
           "ModelShape", "SHAPES", "synth_weights", "FLAVOURS", "LIB_PATH", "HEADER_PATH"]
