"""The C++ host side (kuiperllama_b200/kuiper): the reference's kuiper:: API over libkllm_b200.
(File name: sorts after the kernel / decoder suites, whose parity results it builds on.)

not gpu: it builds with CMake, the reference's demo/main.cpp and demo/main_qwen.cpp compile and
         link against it UNCHANGED (when KUIPER_REFERENCE_DIR names a reference checkout), and it
         fails loudly without a GPU.
gpu:     decoding through model::LLama2Model / Qwen2Model (the demo's embedding -> fill_input ->
         predict loop) reproduces the committed goldens and is bit-identical to the C-ABI decoder,
         on the fused path and on the layer-by-layer op-registry path.
"""
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT as REPO

sys.path.insert(0, str(REPO / "kuiperllama_b200" / "kuiper"))
import build_host  # noqa: E402

REFERENCE_PRESENT = build_host.reference_checkout() is not None
TOL = 1e-4


def ensure_built(variant):
    exe = build_host.binary(variant, "kuiper_decode")
    if not exe.exists():
        build_host.build(variant)
    return exe


def run_decode(variant, checkpoint, family, prec, n_steps, ids, layers=False, logits=None, env=None, copy_at=None):
    cmd = [str(ensure_built(variant)), str(checkpoint), family, prec, str(n_steps), *map(str, ids)]
    if layers:
        cmd.append("--layers")
    if copy_at is not None:
        cmd += ["--copy-at", str(copy_at)]
    if logits is not None:
        cmd += ["--logits", str(logits)]
    return subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=env)


@pytest.mark.parametrize("variant", ["llama2", "qwen2"])
def test_host_library_builds_and_reference_demos_link_unchanged(kllm_lib, variant):
    out = build_host.build(variant)
    assert (out / "libllama.so").exists()
    assert (out / "kuiper_decode").exists()
    if REFERENCE_PRESENT:
        assert (out / "llama_infer").exists(), "reference demo/main.cpp did not build against our headers"
        if variant == "qwen2":
            assert (out / "qwen_infer").exists(), "reference demo/main_qwen.cpp did not build"
    # every kuiper:: symbol the demos need resolves inside libllama.so / libkllm_b200.so
    ldd = subprocess.run(["ldd", str(out / "kuiper_decode")], capture_output=True, text=True).stdout
    assert "not found" not in ldd, ldd
    assert "libkllm_b200.so" in ldd


def test_host_api_selftest_cpu_cases(kllm_lib):
    """tools/kuiper_selftest.cpp: the CPU cases of the reference's gtest programs for Buffer / Tensor
    (test/test_tensor/*.cpp) plus Status, layer check() and checkpoint-header behaviour."""
    out = build_host.build("llama2")
    r = subprocess.run([str(out / "kuiper_selftest"), str(GOLDEN / "tiny_llama2_fp32.bin")], capture_output=True,
                       text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "0 failed expectation(s)" in r.stdout and "FAILED" not in r.stdout


@pytest.mark.parametrize("name,family,prec", [("tiny_llama2_fp32", "llama", "fp32"),
                                              ("tiny_llama2_fp32_shared", "llama", "fp32"),
                                              ("tiny_llama2_int8", "llama", "int8"),
                                              ("tiny_qwen2file_fp32", "qwen", "fp32")])
def test_host_loading_pipeline_without_a_gpu(kllm_lib, name, family, prec):
    """Model::gen_model_from_file on the golden checkpoints (no init(), no GPU): header -> config, and
    every layer's weight / scale / bias is a view into the mapping at the offset the exporter's
    layout implies (computed independently inside kuiper_selftest)."""
    out = build_host.build("llama2")
    r = subprocess.run([str(out / "kuiper_selftest"), str(GOLDEN / f"{name}.bin"), family, prec],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "[  ok  ] model loading pipeline" in r.stdout and "0 failed expectation(s)" in r.stdout


def test_host_fails_loudly_without_a_gpu(kllm_lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = run_decode("llama2", GOLDEN / "tiny_llama2_fp32.bin", "llama", "fp32", 2, [1])
    assert r.returncode != 0
    assert "CUDA" in r.stderr


def test_host_rejects_cpu_device_and_truncated_checkpoints(kllm_lib, tmp_path):
    """init(kDeviceCPU) and a file shorter than its header implies are errors, not crashes."""
    blob = (GOLDEN / "tiny_llama2_fp32.bin").read_bytes()
    short = tmp_path / "short.bin"
    short.write_bytes(blob[: len(blob) // 2])
    r = run_decode("llama2", short, "llama", "fp32", 2, [1])
    assert r.returncode != 0 and r.returncode > 0, r  # clean exit code, not a signal


GOLDENS = [("tiny_llama2_fp32", "llama", "fp32", False, "llama2"),
           ("tiny_llama2_fp32_shared", "llama", "fp32", False, "llama2"),
           ("tiny_llama2_int8", "llama", "int8", True, "llama2"),
           # qwen FILE layout (q/k/v biases) with llama2 arithmetic = Qwen2Model in a default build
           ("tiny_qwen2file_fp32", "qwen", "fp32", False, "llama2")]


@pytest.mark.gpu
@pytest.mark.parametrize("layers", [False, True], ids=["fused", "layers"])
@pytest.mark.parametrize("name,family,prec,quant,variant", GOLDENS)
def test_cpp_model_matches_goldens_and_cabi(kllm_lib, tmp_path, name, family, prec, quant, variant, layers):
    from test_decoder_gpu import load_decoder
    g = np.load(GOLDEN / f"{name}.npz")
    toks = [int(t) for t in g["tokens"]]
    out = tmp_path / "logits.f32"
    r = run_decode(variant, GOLDEN / f"{name}.bin", family, prec, len(toks), toks, layers=layers, logits=out)
    assert r.returncode == 0, r.stderr
    chosen = [int(x) for x in r.stdout.split()]
    logits = np.fromfile(out, dtype=np.float32)
    want = g["logits"][len(toks) - 1]
    assert np.abs(logits - want).max() < TOL
    assert chosen[:-1] == [-1] * (len(toks) - 1) and chosen[-1] == int(np.argmax(want))
    # bit-identical to the C-ABI decoder fed the same tokens
    dec, _ = load_decoder(GOLDEN / f"{name}.bin", quant, "llama2", family == "qwen")
    for t, tok in enumerate(toks):
        nxt = dec.step(tok, t)
    assert nxt == chosen[-1]
    assert np.array_equal(dec.logits().view(np.uint32), logits.view(np.uint32))
    dec.close()


@pytest.mark.gpu
@pytest.mark.parametrize("key,variant,family,prec", [("small", "llama2", "llama", "fp32"),
                                                     ("small-int8", "llama2", "llama", "int8"),
                                                     ("small-qwen", "qwen2", "qwen", "fp32")])
def test_cpp_free_running_decode_identical_to_cabi(kllm_lib, tmp_path, key, variant, family, prec):
    """The demo loop (prompt of 3 ids, then greedy) through the C++ model == the C-ABI decoder,
    on both host paths."""
    from kuiperllama_b200 import SHAPES, Decoder, synth_weights
    from kuiperllama_b200.checkpoint import write_checkpoint
    shape = SHAPES[key]
    w = synth_weights(shape, "cuda", 77)
    path = tmp_path / f"{key}.bin"
    write_checkpoint(str(path), shape, w)
    prompt, steps = [1, 5, 9], 40
    dec = Decoder(shape, w)
    want, tok = [], None
    for pos in range(steps):
        tok = dec.step(prompt[pos] if pos < len(prompt) else tok, pos, pos < len(prompt) - 1)
        want.append(tok)
    want = want[len(prompt) - 1:]
    for layers in (False, True):
        r = run_decode(variant, path, family, prec, steps, prompt, layers=layers)
        assert r.returncode == 0, r.stderr
        chosen = [int(x) for x in r.stdout.split()]
        assert chosen[len(prompt) - 1:] == want, ("layers" if layers else "fused")
    dec.close()


@pytest.mark.gpu
@pytest.mark.parametrize("copy_at", [0, 3, 9])
def test_cpp_predict_keeps_one_history_when_a_step_leaves_the_fused_decoder(kllm_lib, tmp_path, copy_at):
    """predict() runs in the fused decoder when it recognises its input as an embedding() row and
    layer by layer otherwise; the two keep separate KV caches.  A sequence that leaves the decoder in
    the middle (position K gets a COPY of the row) must still attend over the whole history: the
    decoder's rows are copied into the layer path's cache, later positions stay on the layer path.
    Ids and final logits are bit-identical to the uninterrupted fused run."""
    name = "tiny_llama2_fp32"
    g = np.load(GOLDEN / f"{name}.npz")
    toks = [int(t) for t in g["tokens"]][:4]
    n = 14
    a, b = tmp_path / "a.f32", tmp_path / "b.f32"
    r0 = run_decode("llama2", GOLDEN / f"{name}.bin", "llama", "fp32", n, toks, logits=a)
    r1 = run_decode("llama2", GOLDEN / f"{name}.bin", "llama", "fp32", n, toks, logits=b, copy_at=copy_at)
    assert r0.returncode == 0 and r1.returncode == 0, r0.stderr + r1.stderr
    assert r0.stdout.split() == r1.stdout.split()
    assert np.array_equal(np.fromfile(a, dtype=np.uint32), np.fromfile(b, dtype=np.uint32))
