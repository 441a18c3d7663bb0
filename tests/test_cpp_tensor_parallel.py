"""Tensor parallelism of the C++ host side (kuiper/include/model/tensor_parallel.h): one process per GPU,
no torch, no MPI.

not gpu: the shard rules equal the Python side's (kuiperllama_b200/tensor_parallel.py), the TCP rendezvous
         gathers every rank's blob on every rank (world 2, 4, 8), and the LOAD-TIME sharding of
         LLama2Model / Qwen2Model -- row slices viewed in the mmap, column slices packed into staging
         buffers, int8 group scales and Qwen2 biases following -- yields byte for byte what shard_weights()
         cuts out of the same checkpoint (FNV-1a hashes printed by tools/kuiper_tp_check.cpp).
gpu:     (needs >= 2 GPUs) `kuiper_tp_launch 2 kuiper_decode ...` decodes the same ids as the single-GPU run.
"""
import socket
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT as REPO

sys.path.insert(0, str(REPO / "kuiperllama_b200" / "kuiper"))
import build_host  # noqa: E402

from kuiperllama_b200 import tensor_parallel as tp  # noqa: E402
from kuiperllama_b200.checkpoint import write_checkpoint  # noqa: E402
from kuiperllama_b200.decoder import ModelShape, synth_weights  # noqa: E402


def tool(variant, name):
    exe = build_host.binary(variant, name)
    if not exe.exists():
        build_host.build(variant)
    return str(exe)


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


SHAPES = {
    "tinyllama": ModelShape("tinyllama", 2048, 5632, 22, 32, 4, 32000, 2048),
    "llama2-7b-int8": ModelShape("l7b8", 4096, 11008, 32, 32, 32, 32000, 2048, group_size=64),
    "qwen2.5-0.5b": ModelShape("qwen", 896, 4864, 24, 14, 2, 151936, 32768, flavour="qwen2"),
    "small-int8": ModelShape("s8", 256, 1024, 2, 4, 2, 512, 64, group_size=64),
}


@pytest.mark.parametrize("key", sorted(SHAPES))
@pytest.mark.parametrize("world", [1, 2, 4, 8])
def test_shard_rules_equal_python(kllm_lib, key, world):
    s = SHAPES[key]
    try:
        tp.check_shardable(s, world)
        ok = True
    except Exception:
        ok = False
    for rank in range(world):
        r = subprocess.run([tool("llama2", "kuiper_tp_check"), "shard", *map(str, (
            s.dim, s.hidden_dim, s.layer_num, s.head_num, s.kv_head_num, s.vocab_size, s.group_size, world, rank))],
            capture_output=True, text=True, timeout=60)
        if not ok:
            assert r.returncode == 3 and r.stdout.startswith("error"), (r.stdout, r.stderr)
            continue
        assert r.returncode == 0, (r.stdout, r.stderr)
        f = r.stdout.split()
        got = {f[0]: (int(f[1]), int(f[2])), f[3]: (int(f[4]), int(f[5])), f[6]: (int(f[7]), int(f[8])),
               "heads": int(f[10]), "kv_heads": int(f[12]), "hidden": int(f[14]), "comm_words": int(f[16])}
        hs = s.head_size
        kvh = tp.kv_heads_of_rank(s, world, rank)
        ffn = tp.ffn_range(s, world, rank)
        loc = tp.local_shape(s, world, rank) if world > 1 else s
        assert got["q"] == (rank * (s.head_num // world) * hs, (rank + 1) * (s.head_num // world) * hs)
        assert got["k"] == (kvh.start * hs, kvh.stop * hs)
        assert got["f"] == (ffn.start, ffn.stop)
        assert (got["heads"], got["kv_heads"], got["hidden"]) == (loc.head_num, loc.kv_head_num, loc.hidden_dim)
        assert got["comm_words"] == (tp.comm_words(s, world) + 3) // 4 * 4


@pytest.mark.parametrize("world", [2, 4, 8])
def test_rendezvous_gathers_on_every_rank(kllm_lib, world):
    port = free_port()
    exe = tool("llama2", "kuiper_tp_check")
    procs = [subprocess.Popen([exe, "rendezvous", str(world), str(r), str(port)], stdout=subprocess.PIPE,
                              stderr=subprocess.PIPE, text=True) for r in reversed(range(world))]  # rank 0 starts LAST
    for p in procs:
        out, err = p.communicate(timeout=90)
        assert p.returncode == 0, (out, err)
        assert ": ok" in out


def fnv1a(b: bytes) -> int:
    # vectorised FNV-1a would need 64-bit wraparound per byte; the shards here are small
    h = 1469598103934665603
    for c in b:
        h = ((h ^ c) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return h


LOAD_CASES = {
    # key: (shape, family, precision, build variant)
    "fp32": (ModelShape("tp-fp32", 128, 384, 2, 4, 2, 96, 32), "llama", "fp32", "llama2"),
    "fp32-kv-replicated": (ModelShape("tp-kvrep", 128, 256, 2, 4, 1, 96, 32), "llama", "fp32", "llama2"),
    "int8": (ModelShape("tp-int8", 256, 768, 2, 4, 2, 96, 32, group_size=64), "llama", "int8", "llama2"),
    "qwen-bias": (ModelShape("tp-qwen", 128, 384, 2, 4, 2, 96, 32, flavour="qwen2"), "qwen", "fp32", "qwen2"),
    # 8 heads over 2 kv heads: at world 8 four ranks share each kv head (TinyLlama's situation at 8 GPUs)
    "fp32-gqa8": (ModelShape("tp-gqa8", 256, 512, 2, 8, 2, 96, 32), "llama", "fp32", "llama2"),
    "int8-gqa8": (ModelShape("tp-int8-gqa8", 512, 2048, 2, 8, 2, 96, 32, group_size=64), "llama", "int8", "llama2"),
}


@pytest.mark.parametrize("key", sorted(LOAD_CASES))
@pytest.mark.parametrize("world", [2, 4, 8])
def test_load_time_sharding_equals_shard_weights(kllm_lib, tmp_path, key, world):
    shape, family, prec, variant = LOAD_CASES[key]
    try:
        tp.check_shardable(shape, world)
    except Exception:
        pytest.skip(f"{shape.name} does not split {world} ways")
    w = synth_weights(shape, device="cpu", seed=7)
    path = tmp_path / f"{shape.name}.bin"
    write_checkpoint(str(path), shape, w)
    exe = tool(variant, "kuiper_tp_check")
    for rank in range(world):
        r = subprocess.run([exe, "load", str(path), family, prec, str(world), str(rank)], capture_output=True,
                           text=True, timeout=120)
        assert r.returncode == 0, (r.stdout, r.stderr)
        shard = tp.shard_weights(shape, w, world, rank)
        loc = tp.local_shape(shape, world, rank)
        lines = [ln.split() for ln in r.stdout.strip().splitlines()]
        assert lines[-1] == ["local", "heads", str(loc.head_num), "kv_heads", str(loc.kv_head_num), "hidden",
                             str(loc.hidden_dim)]
        seen = 0
        for f in lines[:-1]:
            name, layer = f[0], int(f[1])
            arr = np.ascontiguousarray(shard[name][layer].numpy() if hasattr(shard[name], "numpy") else shard[name][layer])
            assert (int(f[3]), int(f[4])) == tuple(arr.shape), (name, layer, f, arr.shape)
            assert int(f[6], 16) == fnv1a(arr.tobytes()), f"{name}[{layer}] of rank {rank}: weight bytes differ"
            rest = f[7:]
            if prec == "int8":
                sc = shard["s" + name[1:]][layer]
                sc = np.ascontiguousarray(sc.numpy() if hasattr(sc, "numpy") else sc)
                assert rest[0] == "s" and int(rest[1]) == sc.size
                assert int(rest[2], 16) == fnv1a(sc.tobytes()), f"{name}[{layer}] of rank {rank}: scales differ"
                rest = rest[3:]
            if rest:
                b = shard["b" + name[1:]][layer]
                b = np.ascontiguousarray(b.numpy() if hasattr(b, "numpy") else b)
                assert rest[0] == "b" and int(rest[1]) == b.size
                assert int(rest[2], 16) == fnv1a(b.tobytes()), f"{name}[{layer}] of rank {rank}: bias differs"
            seen += 1
        assert seen == 7 * shape.layer_num


def test_launcher_sets_the_environment_and_propagates_failure(kllm_lib):
    exe = tool("llama2", "kuiper_tp_launch")
    r = subprocess.run([exe, "2", "--all-stdout", "--port", "31000", "--", "sh", "-c",
                        "echo $KUIPER_TP_WORLD $KUIPER_TP_RANK $KUIPER_TP_PORT $KUIPER_TP_DEVICE"],
                       capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stderr
    assert sorted(r.stdout.strip().splitlines()) == ["2 0 31000 0", "2 1 31000 1"]
    r = subprocess.run([exe, "2", "--", "sh", "-c", "echo rank $KUIPER_TP_RANK"], capture_output=True, text=True,
                       timeout=60)
    assert r.stdout.strip() == "rank 0"  # the other ranks' stdout is dropped
    r = subprocess.run([exe, "2", "--", "sh", "-c", "if [ $KUIPER_TP_RANK = 1 ]; then exit 7; else sleep 30; fi"],
                       capture_output=True, text=True, timeout=25)
    assert r.returncode == 7  # and rank 0 did not keep the launcher for its 30 seconds


def _need_gpus(n):
    import torch
    if torch.cuda.device_count() < n:
        pytest.skip(f"needs {n} GPUs")


@pytest.mark.gpu
@pytest.mark.parametrize("key,family,prec,variant", [("small-tp", "llama", "fp32", "llama2"),
                                                     ("small-tp-int8", "llama", "int8", "llama2"),
                                                     ("small-qwen", "qwen", "fp32", "qwen2")])
@pytest.mark.parametrize("world", [2, 4])
def test_cpp_tensor_parallel_decode_equals_single_gpu(kllm_lib, tmp_path, key, family, prec, variant, world):
    """kuiper_tp_launch N kuiper_decode: N processes, each loading its shard of the checkpoint in C++ and
    meeting over the TCP rendezvous + CUDA-IPC, decode the same greedy ids as one GPU (both runs in the exact
    numerics; the split changes the summation tree of wo / w2, so logits agree to 1e-4, ids wherever the
    top-2 margin allows -- these seeds keep a margin)."""
    _need_gpus(world)
    from kuiperllama_b200 import SHAPES
    shape = SHAPES[key]
    try:
        tp.check_shardable(shape, world)
    except Exception:
        pytest.skip(f"{shape.name} does not split {world} ways")
    w = synth_weights(shape, device="cpu", seed=11)
    path = tmp_path / "model.bin"
    write_checkpoint(str(path), shape, w)
    steps, prompt = 40, [1, 5, 9]
    decode = tool(variant, "kuiper_decode")
    one = subprocess.run([decode, str(path), family, prec, str(steps), *map(str, prompt), "--logits",
                          str(tmp_path / "one.f32")], capture_output=True, text=True, timeout=300)
    assert one.returncode == 0, one.stderr
    many = subprocess.run([tool(variant, "kuiper_tp_launch"), str(world), "--port", str(free_port()), "--", decode,
                           str(path), family, prec, str(steps), *map(str, prompt), "--logits",
                           str(tmp_path / "tp.f32")], capture_output=True, text=True, timeout=600)
    assert many.returncode == 0, many.stderr
    assert "persistent" in many.stderr  # the sharded path is the fused decoder with the tagged exchange
    a = np.fromfile(tmp_path / "one.f32", np.float32)
    b = np.fromfile(tmp_path / "tp.f32", np.float32)
    assert a.shape == b.shape == (shape.vocab_size,)
    assert np.abs(a - b).max() < 1e-4
    assert one.stdout.split() == many.stdout.split()
