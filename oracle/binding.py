"""ctypes bindings for the two checkers:

  Oracle     oracle/_build/liboracle.so      plain-C restatement of the reference CPU path
  RefCuda    oracle/_ref/libkuiper_ref.so    the reference's own sources compiled for sm_100a
             (+ libkuiper_ref_qwen2_kernels.so: its kernels under -DQWEN2_SUPPORT)

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_int8, c_void_p
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ORACLE_SO = HERE / "_build" / "liboracle.so"
REF_SO = HERE / "_ref" / "libkuiper_ref.so"
REF_QWEN_SO = HERE / "_ref" / "libkuiper_ref_qwen2_kernels.so"

FLAVOURS = {"llama2": 0, "llama3": 1, "qwen2": 2, "qwen2file": 3}


def reference_tree() -> Path | None:
    """The reference checkout named by KUIPER_REFERENCE_DIR, or None when the variable is unset or
    the tree cannot be read (an unreadable path is the same as an absent one)."""
    d = os.environ.get("KUIPER_REFERENCE_DIR")
    if not d:
        return None
    try:
        return Path(d) if (Path(d) / "kuiper" / "source").is_dir() else None
    except OSError:
        return None


def build_oracle() -> Path:
    subprocess.check_call(["make", "-s", "-C", str(HERE), "oracle"])
    return ORACLE_SO


def build_ref(jobs: int = 8) -> bool:
    """Compile oracle/_ref from the reference checkout when KUIPER_REFERENCE_DIR names one;
    otherwise report whether an earlier build of oracle/_ref is present."""
    tree = reference_tree()
    if tree is None:
        return REF_SO.exists()
    subprocess.check_call(["make", "-s", f"-j{jobs}", "-C", str(HERE), f"REF={tree}", "ref"])
    return True


def _f32(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a, a.ctypes.data_as(POINTER(c_float))


class KoConfig(ctypes.Structure):
    _fields_ = [(n, c_int32) for n in (
        "dim", "hidden_dim", "layer_num", "head_num", "kv_head_num", "vocab_size", "seq_len",
        "kv_dim", "kv_mul", "head_size", "shared_classifier", "is_quant", "group_size", "flavour")]


class Oracle:
    """numpy front-end of kuiper_oracle.c (each method cites the C function it calls)."""

    def __init__(self):
        if not ORACLE_SO.exists():
            build_oracle()
        L = ctypes.CDLL(str(ORACLE_SO))
        fp = POINTER(c_float)
        L.ko_matmul_f32.argtypes = [fp, fp, fp, c_int, c_int, c_float]
        L.ko_matmul_f32_cuda_order.argtypes = [fp, fp, fp, c_int, c_int]
        L.ko_matmul_w8.argtypes = [fp, POINTER(c_int8), fp, fp, c_int, c_int, c_int]
        L.ko_matmul_w8_cuda_order.argtypes = [fp, POINTER(c_int8), fp, fp, c_int, c_int, c_int]
        L.ko_rmsnorm.argtypes = [fp, fp, fp, c_int, c_float]
        L.ko_add.argtypes = [fp, fp, fp, c_int]
        L.ko_swiglu.argtypes = [fp, fp, fp, c_int]
        L.ko_softmax_inplace.argtypes = [fp, c_int]
        L.ko_embedding.argtypes = [POINTER(c_int32), c_int, fp, fp, c_int, c_int]
        L.ko_argmax.argtypes = [fp, c_int64]
        L.ko_argmax.restype = c_int64
        L.ko_sincos.argtypes = [c_int, c_int, c_float, fp, fp]
        L.ko_rope.argtypes = [c_int, c_int, c_int, c_int, fp, fp, c_int, fp, fp]
        L.ko_mha.argtypes = [c_int] * 7 + [fp, fp, fp, fp, fp]
        L.ko_quantize_q80.argtypes = [fp, c_int64, c_int, POINTER(c_int8), fp]
        L.ko_flavour_eps.restype = c_float
        L.ko_flavour_eps.argtypes = [c_int]
        L.ko_flavour_theta.restype = c_float
        L.ko_flavour_theta.argtypes = [c_int]
        L.ko_set_matmul_mode.argtypes = [c_int]
        L.ko_set_blas_library.argtypes = [c_char_p]
        L.ko_num_threads.restype = c_int
        L.ko_set_num_threads.restype = c_int
        L.ko_set_num_threads.argtypes = [c_int]
        L.ko_model_open.restype = c_void_p
        L.ko_model_open.argtypes = [c_char_p, c_int, c_int]
        L.ko_model_close.argtypes = [c_void_p]
        L.ko_model_config.restype = POINTER(KoConfig)
        L.ko_model_config.argtypes = [c_void_p]
        L.ko_model_step.argtypes = [c_void_p, c_int, c_int, fp]
        L.ko_model_key_cache.restype = fp
        L.ko_model_key_cache.argtypes = [c_void_p]
        L.ko_model_value_cache.restype = fp
        L.ko_model_value_cache.argtypes = [c_void_p]
        self.L = L

    def eps(self, flavour): return float(self.L.ko_flavour_eps(FLAVOURS[flavour]))
    def theta(self, flavour): return float(self.L.ko_flavour_theta(FLAVOURS[flavour]))

    def matmul(self, x, w, scale=1.0, cuda_order=False):
        x, px = _f32(x); w, pw = _f32(w)
        K, M = w.shape
        out = np.empty(K, np.float32)
        po = out.ctypes.data_as(POINTER(c_float))
        if cuda_order:
            self.L.ko_matmul_f32_cuda_order(px, pw, po, M, K)
        else:
            self.L.ko_matmul_f32(px, pw, po, M, K, scale)
        return out

    def matmul_w8(self, x, q, scales, group, cuda_order=False):
        x, px = _f32(x)
        q = np.ascontiguousarray(q, dtype=np.int8)
        scales, ps = _f32(scales)
        K, M = q.shape
        out = np.empty(K, np.float32)
        fn = self.L.ko_matmul_w8_cuda_order if cuda_order else self.L.ko_matmul_w8
        fn(px, q.ctypes.data_as(POINTER(c_int8)), ps, out.ctypes.data_as(POINTER(c_float)), M, K, group)
        return out

    def quantize_q80(self, w, group):
        w, pw = _f32(w)
        q = np.empty(w.shape, np.int8)
        sc = np.empty(w.size // group, np.float32)
        self.L.ko_quantize_q80(pw, w.size, group, q.ctypes.data_as(POINTER(c_int8)),
                               sc.ctypes.data_as(POINTER(c_float)))
        return q, sc

    def rmsnorm(self, x, w, eps):
        x, px = _f32(x); w, pw = _f32(w)
        out = np.empty_like(x)
        self.L.ko_rmsnorm(px, pw, out.ctypes.data_as(POINTER(c_float)), x.size, eps)
        return out

    def add(self, a, b):
        a, pa = _f32(a); b, pb = _f32(b)
        out = np.empty_like(a)
        self.L.ko_add(pa, pb, out.ctypes.data_as(POINTER(c_float)), a.size)
        return out

    def swiglu(self, a, b):
        a, pa = _f32(a); b, pb = _f32(b)
        out = np.empty_like(a)
        self.L.ko_swiglu(pa, pb, out.ctypes.data_as(POINTER(c_float)), a.size)
        return out

    def softmax(self, x):
        x = np.array(x, dtype=np.float32, copy=True)
        self.L.ko_softmax_inplace(x.ctypes.data_as(POINTER(c_float)), x.size)
        return x

    def embedding(self, tokens, table):
        tokens = np.ascontiguousarray(tokens, dtype=np.int32)
        table, pt = _f32(table)
        vocab, dim = table.shape
        out = np.zeros((tokens.size, dim), np.float32)
        self.L.ko_embedding(tokens.ctypes.data_as(POINTER(c_int32)), tokens.size, pt,
                            out.ctypes.data_as(POINTER(c_float)), dim, vocab)
        return out

    def argmax(self, x):
        x, px = _f32(x)
        return int(self.L.ko_argmax(px, x.size))

    def sincos(self, head_size, seq_len, flavour):
        s = np.empty((seq_len, head_size), np.float32)
        c = np.empty((seq_len, head_size), np.float32)
        self.L.ko_sincos(head_size, seq_len, self.theta(flavour),
                         s.ctypes.data_as(POINTER(c_float)), c.ctypes.data_as(POINTER(c_float)))
        return s, c

    def rope(self, flavour, q, k, pos, sin, cos, head_size):
        q = np.array(q, dtype=np.float32, copy=True); k = np.array(k, dtype=np.float32, copy=True)
        sin, ps = _f32(sin); cos, pc = _f32(cos)
        self.L.ko_rope(FLAVOURS[flavour], q.size, k.size, head_size,
                       q.ctypes.data_as(POINTER(c_float)), k.ctypes.data_as(POINTER(c_float)),
                       pos, ps, pc)
        return q, k

    def mha(self, pos, head_num, layer, seq_len, kv_dim, kv_mul, head_size, q, kc, vc):
        q, pq = _f32(q); kc, pk = _f32(kc); vc, pv = _f32(vc)
        out = np.zeros(head_num * head_size, np.float32)
        score = np.zeros(head_num * seq_len, np.float32)
        self.L.ko_mha(pos, head_num, layer, seq_len, kv_dim, kv_mul, head_size,
                      out.ctypes.data_as(POINTER(c_float)), pq,
                      score.ctypes.data_as(POINTER(c_float)), pk, pv)
        return out, score.reshape(head_num, seq_len)

    # ---- whole model -----------------------------------------------------------------
    def open_model(self, path, is_quant=False, flavour="llama2"):
        h = self.L.ko_model_open(str(path).encode(), int(is_quant), FLAVOURS[flavour])
        if not h:
            raise RuntimeError(f"ko_model_open failed for {path}")
        return OracleModel(self, h)

    def use_fast_matmul(self, on=True, blas=None):
        """Timed-baseline mode only: OpenBLAS sgemv (what Armadillo calls) or OpenMP rows."""
        self.blas_loaded = False
        if on and blas:
            self.blas_loaded = self.L.ko_set_blas_library(str(blas).encode()) == 0
        self.L.ko_set_matmul_mode(1 if on else 0)
        return self.blas_loaded

    def num_threads(self):
        return int(self.L.ko_num_threads())

    def set_num_threads(self, n):
        """OpenMP and the loaded BLAS through their own APIs (survives OMP_NUM_THREADS=1 in the
        environment); returns the thread count the BLAS reports (0: no BLAS loaded)."""
        return int(self.L.ko_set_num_threads(int(n)))


class OracleModel:
    def __init__(self, oracle, handle):
        self.o, self.h = oracle, handle
        self.cfg = oracle.L.ko_model_config(handle).contents

    def step(self, token, pos, want_logits=True):
        buf = np.empty(self.cfg.vocab_size, np.float32) if want_logits else None
        p = buf.ctypes.data_as(POINTER(c_float)) if want_logits else None
        nxt = self.o.L.ko_model_step(self.h, int(token), int(pos), p)
        return nxt, buf

    def kv_cache(self):
        n = self.cfg.layer_num * self.cfg.seq_len * self.cfg.kv_dim
        shape = (self.cfg.layer_num, self.cfg.seq_len, self.cfg.kv_dim)
        k = np.ctypeslib.as_array(self.o.L.ko_model_key_cache(self.h), (n,)).reshape(shape)
        v = np.ctypeslib.as_array(self.o.L.ko_model_value_cache(self.h), (n,)).reshape(shape)
        return k, v

    def close(self):
        if self.h:
            self.o.L.ko_model_close(self.h)
            self.h = None


def find_openblas():
    """A BLAS with cblas_sgemv for the TIMED cpu baseline (the reference's Armadillo would
    call OpenBLAS sgemv).  Bundled in wheels in this image; every candidate is dlopen-ed and
    checked for the symbol (a wheel-bundled library may miss its own dependencies); None if
    nothing usable is found."""
    import glob
    import site
    pats = ["scipy.libs/libscipy_openblas-*.so*", "opencv_python_headless.libs/libopenblas*.so*"]
    for sp in site.getsitepackages():
        for pat in pats:
            for hit in sorted(glob.glob(os.path.join(sp, pat))):
                try:
                    lib = ctypes.CDLL(hit, mode=ctypes.RTLD_LOCAL)
                except OSError:
                    continue
                if hasattr(lib, "cblas_sgemv") or hasattr(lib, "scipy_cblas_sgemv"):
                    return hit
    return None


class RefCuda:
    """The reference's own CUDA kernels / model (oracle/_ref).  Device pointers are plain ints
    (torch .data_ptr())."""

    def __init__(self, flavour="llama2"):
        so = REF_SO if flavour == "llama2" else REF_QWEN_SO
        if not so.exists():
            raise FileNotFoundError(f"{so} not built (run `make -C oracle REF=<reference checkout> ref`)")
        L = ctypes.CDLL(str(so))
        vp = c_void_p
        L.kref_flavour.restype = c_char_p
        L.kref_matmul_f32.argtypes = [vp, vp, vp, c_int, c_int, vp]
        L.kref_matmul_w8.argtypes = [vp, vp, vp, vp, c_int, c_int, c_int, vp]
        L.kref_rmsnorm.argtypes = [vp, vp, vp, c_int, vp]
        L.kref_add.argtypes = [vp, vp, vp, c_int, vp]
        L.kref_swiglu.argtypes = [vp, vp, vp, c_int, vp]
        L.kref_sincos.argtypes = [c_int, c_int, vp, vp, vp]
        L.kref_rope.argtypes = [c_int, c_int, c_int, vp, vp, c_int, vp, vp, c_int, vp]
        L.kref_mha.argtypes = [c_int] * 7 + [vp, vp, vp, vp, vp, c_int, vp]
        L.kref_embedding.argtypes = [POINTER(c_int32), c_int, vp, vp, c_int, c_int, vp]
        L.kref_argmax.argtypes = [vp, c_int64, vp]
        L.kref_argmax.restype = c_int64
        if flavour == "llama2":
            L.kref_model_create.restype = vp
            L.kref_model_create.argtypes = [c_char_p, c_int]
            L.kref_model_destroy.argtypes = [vp]
            L.kref_model_step.argtypes = [vp, c_int, c_int, POINTER(c_float), c_int]
            L.kref_cpu_model_create.restype = vp
            L.kref_cpu_model_create.argtypes = [c_char_p]
            L.kref_cpu_model_destroy.argtypes = [vp]
            L.kref_cpu_model_step.argtypes = [vp, c_int, c_int, POINTER(c_float), c_int]
        self.L = L
        self.flavour = L.kref_flavour().decode()
        assert self.flavour == flavour, (self.flavour, flavour)
