"""ctypes front-end of the device-resident decoder (``kllm_decoder_*``) plus synthetic
random-init weights in the shapes BASELINE.json names.

torch is used here only as plumbing: device memory, RNG for the synthetic checkpoints and
stream handles.  All compute on the decode path happens inside libkllm_b200.so.
"""
from __future__ import annotations

import ctypes
import math
from dataclasses import dataclass, replace

from . import DecoderDesc, FLAVOURS, KllmError, check, load_library


@dataclass(frozen=True)
class ModelShape:
    """Header fields of a KuiperLLama checkpoint (kuiper/include/model/config.h:5-13)."""
    name: str
    dim: int
    hidden_dim: int
    layer_num: int
    head_num: int
    kv_head_num: int
    vocab_size: int
    seq_len: int
    shared_classifier: bool = False
    flavour: str = "llama2"
    group_size: int = 0  # 0 = fp32, 64 = export.py --version 3

    @property
    def head_size(self) -> int:
        return self.dim // self.head_num

    @property
    def kv_dim(self) -> int:
        return self.dim * self.kv_head_num // self.head_num

    @property
    def kv_mul(self) -> int:
        return self.head_num // self.kv_head_num

    def weight_bytes_per_token(self) -> int:
        """ALGORITHMIC bytes one decode step must read (SURVEY.md section 8d): every matmul
        weight once (+ int8 scales), the 2L+1 norm vectors, qkv biases and one embedding row."""
        d, h, L, kv, V = self.dim, self.hidden_dim, self.layer_num, self.kv_dim, self.vocab_size
        numel = L * (2 * d * d + 2 * kv * d + 3 * h * d) + V * d
        wbytes = numel * 4 if self.group_size == 0 else numel + (numel // self.group_size) * 4
        extra = (2 * L + 1) * d * 4 + d * 4
        if self.flavour == "qwen2" and self.group_size == 0:
            extra += L * (d + 2 * kv) * 4
        return wbytes + extra

    def kv_bytes_at(self, pos: int) -> int:
        return 2 * self.layer_num * (pos + 1) * self.kv_dim * 4


SHAPES = {
    # BASELINE.json configs (SURVEY.md section 8 table)
    "stories15m": ModelShape("stories15M-fp32", 288, 768, 6, 6, 6, 32000, 256, True),
    "tinyllama-1.1b": ModelShape("TinyLlama-1.1B-fp32", 2048, 5632, 22, 32, 4, 32000, 2048),
    "llama2-7b-int8": ModelShape("Llama-2-7B-int8-g64", 4096, 11008, 32, 32, 32, 32000, 2048,
                                 group_size=64),
    "qwen2.5-0.5b": ModelShape("Qwen2.5-0.5B-fp32", 896, 4864, 24, 14, 2, 151936, 32768, True,
                               flavour="qwen2"),
    "llama2-7b": ModelShape("Llama-2-7B-fp32", 4096, 11008, 32, 32, 32, 32000, 2048),
    # small shapes for parity tests
    "tiny": ModelShape("tiny-fp32", 64, 172, 2, 4, 2, 512, 64),
    "tiny-shared": ModelShape("tiny-shared-fp32", 64, 172, 2, 4, 4, 512, 64, True),
    "tiny-int8": ModelShape("tiny-int8", 128, 384, 2, 4, 2, 512, 64, group_size=64),
    "tiny-qwen": ModelShape("tiny-qwen2", 128, 344, 2, 4, 2, 640, 96, True, flavour="qwen2"),
    "small": ModelShape("small-fp32", 288, 768, 3, 9, 3, 4096, 160),
    "small-hs48": ModelShape("small-hs48-fp32", 288, 768, 3, 6, 6, 4096, 160),
    "small-int8": ModelShape("small-int8", 256, 768, 2, 4, 2, 1024, 96, group_size=64),
    "small-qwen": ModelShape("small-qwen2", 256, 704, 2, 4, 2, 1536, 128, True, flavour="qwen2"),
    # 8 heads / 2 kv heads: splits 2 ways (kv heads sharded) and 4 ways (kv heads replicated)
    "small-tp": ModelShape("small-tp-fp32", 256, 768, 3, 8, 2, 2048, 128),
    # int8 whose 2-way shards still give the persistent ring 16-byte scale rows
    "small-tp-int8": ModelShape("small-tp-int8", 512, 1536, 2, 8, 4, 1024, 96, group_size=64),
}


def quantize_q80(w, group_size: int):
    """tools/export.py:49-73 quantize_q80 on a torch tensor: symmetric int8 per group of
    `group_size` consecutive elements of the flattened tensor, scale = max|w|/127."""
    import torch
    flat = w.float().reshape(-1, group_size)
    wmax = flat.abs().max(dim=1).values
    scale = wmax / 127.0
    q = torch.round(flat / scale[:, None]).to(torch.int8)
    return q.reshape(w.shape), scale.contiguous()


def synth_weights(shape: ModelShape, device="cuda", seed: int = 1234, norm_jitter: float = 0.1):
    """Random-init weights following tools/model.py:233-247 (N(0,0.02^2); wo and w3 scaled by
    1/sqrt(2L)), generated on `device`.  Norm weights are 1 + U(-j, j) so the norm multiply is
    actually exercised.  Returns a dict of contiguous torch tensors (int8 + scales if quant)."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    s = shape
    L, d, h, kv, V = s.layer_num, s.dim, s.hidden_dim, s.kv_dim, s.vocab_size

    def normal(*dims, std=0.02):
        return torch.empty(*dims, device=device, dtype=torch.float32).normal_(0.0, std, generator=g)

    def norm_w(*dims):
        w = torch.ones(*dims, device=device, dtype=torch.float32)
        if norm_jitter:
            w += (torch.rand(*dims, device=device, generator=g) * 2 - 1) * norm_jitter
        return w

    small = 0.02 / math.sqrt(2 * L)
    w = {
        "tok_emb": normal(V, d),
        "attn_norm": norm_w(L, d), "ffn_norm": norm_w(L, d), "final_norm": norm_w(d),
        "wq": normal(L, d, d), "wk": normal(L, kv, d), "wv": normal(L, kv, d),
        "wo": normal(L, d, d, std=small),
        "w1": normal(L, h, d), "w2": normal(L, d, h), "w3": normal(L, h, d, std=small),
    }
    w["wcls"] = None if s.shared_classifier else normal(V, d)
    if s.flavour == "qwen2" and s.group_size == 0:
        w["bq"], w["bk"], w["bv"] = normal(L, d), normal(L, kv), normal(L, kv)
    if s.group_size:
        if s.shared_classifier:
            raise KllmError("int8 + shared classifier is a reference defect (llama3.cpp:259-277)")
        for name in ("wq", "wk", "wv", "wo", "w1", "w2", "w3", "wcls"):
            qs = [quantize_q80(t, s.group_size) for t in (w[name] if name != "wcls" else [w[name]])]
            q = torch.stack([a for a, _ in qs])
            sc = torch.stack([b for _, b in qs])
            if name == "wcls":
                q, sc = q[0], sc[0]
            w[name], w["s" + name[1:]] = q.contiguous(), sc.contiguous()
    return w


def _ptr_array(tensors):
    arr = (ctypes.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])
    return arr


class Decoder:
    """Owns a ``kllm_decoder`` built over torch-held device weights."""

    def __init__(self, shape: ModelShape, weights: dict, stream=None, tp_size=1, tp_rank=0,
                 allreduce=None, allreduce_ctx=None, full_dim=None, comm=None, numerics="exact"):
        self.lib = load_library()
        self.shape = shape
        self.weights = weights  # keep the tensors alive
        s = shape
        L = s.layer_num
        d = DecoderDesc()
        d.dim = full_dim or s.dim
        d.hidden_dim, d.layer_num = s.hidden_dim, L
        d.head_num, d.kv_head_num = s.head_num, s.kv_head_num
        d.vocab_size, d.seq_len = s.vocab_size, s.seq_len
        d.flavour = FLAVOURS[s.flavour]
        d.group_size = s.group_size
        self._keep = []

        def per_layer(t):
            arr = _ptr_array([t[l] for l in range(L)])
            self._keep.append(arr)
            return ctypes.cast(arr, ctypes.POINTER(ctypes.c_void_p))

        d.tok_emb = weights["tok_emb"].data_ptr()
        d.attn_norm, d.ffn_norm = per_layer(weights["attn_norm"]), per_layer(weights["ffn_norm"])
        d.final_norm = weights["final_norm"].data_ptr()
        for n in ("wq", "wk", "wv", "wo", "w1", "w2", "w3"):
            setattr(d, n, per_layer(weights[n]))
        wcls = weights.get("wcls")
        d.wcls = (wcls if wcls is not None else weights["tok_emb"]).data_ptr()
        if s.group_size:
            for n in ("sq", "sk", "sv", "so", "s1", "s2", "s3"):
                setattr(d, n, per_layer(weights[n]))
            d.scls = weights["scls"].data_ptr()
        if "bq" in weights:
            d.bq, d.bk, d.bv = (per_layer(weights[n]) for n in ("bq", "bk", "bv"))
        d.tp_size, d.tp_rank = tp_size, tp_rank
        # "exact": bit-identical to the reference; "fast": toleranced (kllm_b200.h, kllm_decoder_desc::numerics)
        d.numerics = {"exact": 0, "fast": 1}[numerics]
        if allreduce is not None:
            d.allreduce = allreduce
            d.allreduce_ctx = allreduce_ctx
        if comm is not None:
            d.comm = comm.handle
            self.comm = comm  # keep alive
        self.desc = d
        # local head geometry (head counts in `shape` are per-rank under tensor parallelism)
        self.head_size = d.dim // (s.head_num * max(tp_size, 1))
        self.local_kv_dim = s.kv_head_num * self.head_size
        handle = ctypes.c_void_p()
        stream_ptr = ctypes.c_void_p(stream) if stream else None
        check(self.lib.kllm_decoder_create(ctypes.byref(d), stream_ptr, ctypes.byref(handle)),
              "kllm_decoder_create")
        self.handle = handle

    def close(self):
        if getattr(self, "handle", None):
            self.lib.kllm_decoder_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launches_per_step(self) -> int:
        return self.lib.kllm_decoder_launches_per_step(self.handle)

    @property
    def classifier_rows(self) -> int:
        """Classifier rows this rank streams per token (vocab / tp when sharded by vocabulary)."""
        return self.lib.kllm_decoder_classifier_rows(self.handle)

    @property
    def engine(self) -> str:
        return self.lib.kllm_decoder_engine(self.handle).decode()

    def step(self, token: int, pos: int, is_prompt: bool = False) -> int:
        """Reference-facing call with host buffers (predict + post_processing)."""
        nxt = ctypes.c_int32(-1)
        check(self.lib.kllm_decoder_step(self.handle, token, pos, int(is_prompt), ctypes.byref(nxt)),
              "kllm_decoder_step")
        return nxt.value

    def prompt(self, tokens, start_pos: int = 0) -> int:
        """Feed a whole prompt (one launch on the persistent engine, classifier only for the last
        position); returns the greedy id that follows the prompt."""
        n = len(tokens)
        arr = (ctypes.c_int32 * n)(*[int(t) for t in tokens])
        nxt = ctypes.c_int32(-1)
        check(self.lib.kllm_decoder_prompt(self.handle, arr, n, start_pos, ctypes.byref(nxt)), "kllm_decoder_prompt")
        return nxt.value

    def prefill_tf32(self, tokens, start_pos: int = 0) -> int:
        """TOLERANCED batched prefill on the tcgen05 tensor cores (TF32); same contract as prompt()."""
        n = len(tokens)
        arr = (ctypes.c_int32 * n)(*[int(t) for t in tokens])
        nxt = ctypes.c_int32(-1)
        check(self.lib.kllm_decoder_prefill_tf32(self.handle, arr, n, start_pos, ctypes.byref(nxt)),
              "kllm_decoder_prefill_tf32")
        return nxt.value

    def prefill_w8(self, tokens, start_pos: int = 0) -> int:
        """TOLERANCED batched prefill of an int8 (group 64) checkpoint on the tcgen05 kind::i8 tensor cores;
        same contract as prompt(), logits within 1e-4 of it.  Raises KllmError for fp32 checkpoints."""
        n = len(tokens)
        arr = (ctypes.c_int32 * n)(*[int(t) for t in tokens])
        nxt = ctypes.c_int32(-1)
        check(self.lib.kllm_decoder_prefill_w8(self.handle, arr, n, start_pos, ctypes.byref(nxt)),
              "kllm_decoder_prefill_w8")
        return nxt.value

    def generate(self, first_token: int, start_pos: int, n_steps: int, teacher=None):
        out = (ctypes.c_int32 * n_steps)()
        tf = None
        if teacher is not None:
            tf = (ctypes.c_int32 * n_steps)(*[int(t) for t in teacher[:n_steps]])
        check(self.lib.kllm_decoder_generate(self.handle, first_token, start_pos, n_steps, tf, out),
              "kllm_decoder_generate")
        return list(out)

    def logits(self):
        import numpy as np
        buf = np.empty(self.shape.vocab_size, dtype=np.float32)
        check(self.lib.kllm_decoder_logits(self.handle, buf.ctypes.data_as(ctypes.c_void_p)),
              "kllm_decoder_logits")
        return buf

    def kv_cache(self):
        """(key, value) caches as numpy arrays [L, seq_len, kv_dim] in the reference layout."""
        import numpy as np
        s = self.shape
        k = np.empty((s.layer_num, s.seq_len, self.local_kv_dim), np.float32)
        v = np.empty_like(k)
        check(self.lib.kllm_decoder_read_kv(self.handle, k.ctypes.data_as(ctypes.c_void_p),
                                            v.ctypes.data_as(ctypes.c_void_p)), "kllm_decoder_read_kv")
        return k, v
