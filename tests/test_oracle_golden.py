"""Pin the CPU oracle (oracle/kuiper_oracle.c) before trusting it -- SURVEY.md section 8c.

1. every known-answer vector the reference's own tests hold for the path;
2. fixtures produced by importing the reference's PyTorch model + exporters
   (tests/golden/make_golden.py);
3. the reference's own orchestration (llama3.cpp compiled unmodified into oracle/_ref) driving
   the restated kernels must agree with ko_model_step bit for bit (live when oracle/_ref is built,
   and always against its recorded outputs, tests/reference_outputs.py).
"""
import struct

import numpy as np
import pytest

from conftest import GOLDEN
from reference_outputs import check, live_reference


# ---- 1. reference unit-test known answers ---------------------------------------------------
def test_matmul_known_answer_test_load(oracle):
    # test/test_op/test_load.cpp:74-105: W = arange(16*128).reshape(16,128), x = ones(128)
    w = np.arange(16 * 128, dtype=np.float32).reshape(16, 128)
    out = oracle.matmul(np.ones(128, np.float32), w)
    assert out[0] == 8128 and out[1] == 24512 and out[14] == 237504 and out[15] == 253888
    assert np.array_equal(out, oracle.matmul(np.ones(128, np.float32), w, cuda_order=True))


def test_matmul_known_answer_linear_course(oracle):
    # test/test_op/test_cu_matmul.cpp:55-75: x = [1,1,-1], W = 1..9 -> [0,3,6]
    w = np.arange(1, 10, dtype=np.float32).reshape(3, 3)
    x = np.array([1, 1, -1], np.float32)
    assert np.array_equal(oracle.matmul(x, w), [0, 3, 6])
    assert np.array_equal(oracle.matmul(x, w, cuda_order=True), [0, 3, 6])


def test_matmul_4x4_arange(oracle):
    # test/test_op/test_cu_matmul.cpp:10-46: input and weight filled with their index
    w = np.arange(16, dtype=np.float32).reshape(4, 4)
    x = np.arange(4, dtype=np.float32)
    expect = (w.astype(np.float64) @ x.astype(np.float64)).astype(np.float32)
    assert np.array_equal(oracle.matmul(x, w), expect)
    assert np.array_equal(oracle.matmul(x, w, cuda_order=True), expect)


def test_embedding_known_answer(oracle):
    # test/test_op/test_cu_emb.cpp:6-31: table = arange(4*512).reshape(4,512), token 1 -> 512+i
    table = np.arange(4 * 512, dtype=np.float32).reshape(4, 512)
    out = oracle.embedding([1], table)
    assert np.array_equal(out[0], 512 + np.arange(512, dtype=np.float32))


def test_add_known_answer(oracle):
    # test/test_op/test_cu_add.cpp:7-27: 2 + 3 = 5 over 32*151 elements
    n = 32 * 151
    assert np.all(oracle.add(np.full(n, 2.0, np.float32), np.full(n, 3.0, np.float32)) == 5.0)


def test_reference_fixture_file_regenerates():
    # tmp/test.bin = header (16,128,256,512,512,4,1024) + arange(2048) fp32  (test_load.cpp:21-23)
    blob = struct.pack("7i", 16, 128, 256, 512, 512, 4, 1024) + np.arange(2048, dtype=np.float32).tobytes()
    assert len(blob) == 8220
    assert (GOLDEN / "reference_tmp_test.bin").read_bytes() == blob  # a copy of the reference's tmp/test.bin


def test_argmax_first_maximum(oracle):
    x = np.array([0.5, 2.0, -1.0, 2.0, 1.0], np.float32)
    assert oracle.argmax(x) == 1  # std::max_element / lowest index on ties


# ---- 2. PyTorch-reference goldens -------------------------------------------------------------
GOLDENS = [("tiny_llama2_fp32_shared", False, "llama2"), ("tiny_llama2_fp32", False, "llama2"),
           ("tiny_llama2_int8", True, "llama2"), ("tiny_qwen2file_fp32", False, "qwen2file")]


@pytest.mark.parametrize("name,quant,flavour", GOLDENS)
def test_model_matches_reference_pytorch(oracle, name, quant, flavour):
    g = np.load(GOLDEN / f"{name}.npz")
    m = oracle.open_model(GOLDEN / f"{name}.bin", quant, flavour)
    try:
        for t, tok in enumerate(g["tokens"]):
            nxt, logits = m.step(int(tok), t)
            # fp32 both sides, different summation orders: 2e-6 absolute on |logits| <= 1.4
            assert np.abs(logits - g["logits"][t]).max() < 2e-6, (name, t)
            assert nxt == int(np.argmax(g["logits"][t]))
    finally:
        m.close()


def test_quantize_q80_reproduces_exporter_bytes(oracle):
    """ko_quantize_q80 on the fp32 fixture's weights must give the int8 fixture's bytes
    (both files were written by the reference exporters from the same PyTorch model)."""
    from kuiperllama_b200.checkpoint import read_checkpoint
    _, wf = read_checkpoint(GOLDEN / "tiny_llama2_fp32.bin", False)
    _, wq = read_checkpoint(GOLDEN / "tiny_llama2_int8.bin", True)
    for name in ("wq", "wk", "wv", "wo", "w1", "w2", "w3"):
        for l in range(wf[name].shape[0]):
            q, s = oracle.quantize_q80(wf[name][l], 64)
            assert np.array_equal(q, wq[name][l]), (name, l)
            assert np.array_equal(s, wq["s" + name[1:]][l]), (name, l)
    q, s = oracle.quantize_q80(wf["wcls"], 64)
    assert np.array_equal(q, wq["wcls"]) and np.array_equal(s, wq["scls"])


def test_torch_quantizer_matches_oracle(oracle):
    import torch
    from kuiperllama_b200.decoder import quantize_q80
    g = torch.Generator().manual_seed(3)
    w = torch.empty(96, 128).normal_(0, 0.02, generator=g)
    q, s = quantize_q80(w, 64)
    qo, so = oracle.quantize_q80(w.numpy(), 64)
    assert np.array_equal(q.numpy(), qo) and np.array_equal(s.numpy(), so)


def test_checkpoint_writer_reproduces_exporter_bytes(tmp_path):
    """write_checkpoint(read_checkpoint(golden)) must be byte-identical to what the reference
    exporter wrote (the loader-skipped freqs block is compared to 1e-6)."""
    from kuiperllama_b200.checkpoint import read_checkpoint, write_checkpoint
    for name, quant, flavour in [("tiny_llama2_fp32_shared", False, "llama2"),
                                 ("tiny_llama2_fp32", False, "llama2"),
                                 ("tiny_llama2_int8", True, "llama2"),
                                 ("tiny_qwen2file_fp32", False, "qwen2")]:
        src = GOLDEN / f"{name}.bin"
        shape, w = read_checkpoint(src, quant, flavour)
        out = tmp_path / f"{name}.bin"
        write_checkpoint(str(out), shape, w)
        a, b = np.fromfile(src, np.uint8), np.fromfile(out, np.uint8)
        assert a.size == b.size
        if quant:
            assert np.array_equal(a, b)
        else:
            # locate the freqs block: it sits right after final_norm
            s = shape
            n_before = 7 * 4 + 4 * (s.vocab_size * s.dim + (2 * s.layer_num + 1) * s.dim + s.layer_num * (
                2 * s.dim * s.dim + 2 * s.kv_dim * s.dim + 3 * s.hidden_dim * s.dim))
            if "bq" in w:
                n_before += 4 * s.layer_num * (s.dim + 2 * s.kv_dim)
            n_freq = 4 * s.seq_len * s.head_size
            assert np.array_equal(a[:n_before], b[:n_before])
            assert np.array_equal(a[n_before + n_freq:], b[n_before + n_freq:])
            fa = a[n_before:n_before + n_freq].view(np.float32)
            fb = b[n_before:n_before + n_freq].view(np.float32)
            assert np.abs(fa - fb).max() < 1e-6


# ---- 3. restated kernels under the reference's own orchestration ------------------------------
def test_reference_orchestration_agrees_bitwise(oracle):
    import ctypes
    ref = live_reference("llama2")
    for name in ("tiny_llama2_fp32_shared", "tiny_llama2_fp32"):
        g = np.load(GOLDEN / f"{name}.npz")
        h = ref.L.kref_cpu_model_create(str(GOLDEN / f"{name}.bin").encode()) if ref else None
        assert h or not ref
        m = oracle.open_model(GOLDEN / f"{name}.bin", False, "llama2")
        vocab = m.cfg.vocab_size
        ids, logits, r_ids, r_logits = [], [], [], []
        try:
            for t, tok in enumerate(g["tokens"]):
                nxt, lg = m.step(int(tok), t)
                ids.append(nxt); logits.append(lg)
                if h:
                    buf = np.empty(vocab, np.float32)
                    r_ids.append(ref.L.kref_cpu_model_step(h, int(tok), t,
                                                           buf.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), vocab))
                    r_logits.append(buf)
        finally:
            m.close()
            if h:
                ref.L.kref_cpu_model_destroy(h)
        check(logits, r_logits if h else None, f"cpu_orchestration/{name}/logits", f"{name} logits [position, vocab]")
        check(ids, r_ids if h else None, f"cpu_orchestration/{name}/ids", f"{name} token ids")


# ---- consistency of the two matmul orders ------------------------------------------------------
@pytest.mark.parametrize("M,K", [(288, 17), (2048, 9), (896, 5), (11008, 3)])
def test_cuda_order_close_to_strict(oracle, M, K):
    rng = np.random.default_rng(M + K)
    x = rng.standard_normal(M).astype(np.float32)
    w = (rng.standard_normal((K, M)) * 0.02).astype(np.float32)
    a, b = oracle.matmul(x, w), oracle.matmul(x, w, cuda_order=True)
    exact = w.astype(np.float64) @ x.astype(np.float64)
    assert np.abs(a - exact).max() < 2e-5 and np.abs(b - exact).max() < 2e-5


def test_w8_orders_close(oracle):
    rng = np.random.default_rng(5)
    M, K = 1024, 7
    w = (rng.standard_normal((K, M)) * 0.02).astype(np.float32)
    q, s = oracle.quantize_q80(w, 64)
    x = rng.standard_normal(M).astype(np.float32)
    a = oracle.matmul_w8(x, q, s, 64)
    b = oracle.matmul_w8(x, q, s, 64, cuda_order=True)
    exact = (q.astype(np.float64) * np.repeat(s, 64).reshape(K, M).astype(np.float64)) @ x.astype(np.float64)
    assert np.abs(a - exact).max() < 2e-5 and np.abs(b - exact).max() < 2e-5
