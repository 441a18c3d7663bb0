"""Tensor parallelism (SURVEY.md section 8e).

not gpu: the sharding arithmetic, and a world_size-2 (and 4) gloo run in which every process
         decodes with ITS shard through the oracle's ops and the partial sums meet in
         dist.all_reduce -- logits <= 1e-4 from the unsharded oracle model, identical greedy ids.
gpu (needs >= 2 GPUs): kllm_comm all-reduce (peer memory and NCCL)
         against a host-side sum, 2000 calls back to back; the sharded CUDA decoder against the
         unsharded oracle; peer and NCCL transports agree bit for bit on token ids.
"""
import numpy as np
import pytest

from tp_util import OracleShardModel, numpy_weights, spawn

TOL = 1e-4


def _full_model(key, seed=11):
    from kuiperllama_b200 import SHAPES, synth_weights
    shape = SHAPES[key]
    return shape, synth_weights(shape, "cpu", seed)


@pytest.mark.parametrize("key,tp", [("small-tp", 2), ("small-tp", 4), ("small-int8", 2), ("small-qwen", 2)])
def test_shards_tile_the_full_matrices(key, tp):
    from kuiperllama_b200.tensor_parallel import kv_heads_of_rank, local_shape, shard_weights
    shape, w = _full_model(key)
    w = numpy_weights(w)
    shards = [shard_weights(shape, w, tp, r) for r in range(tp)]
    for name in ("wq", "w1", "w3"):
        assert np.array_equal(np.concatenate([s[name] for s in shards], axis=1), w[name])
    for name in ("wo", "w2"):
        assert np.array_equal(np.concatenate([s[name] for s in shards], axis=2), w[name])
    hs = shape.head_size
    for r, s in enumerate(shards):
        heads = kv_heads_of_rank(shape, tp, r)
        assert np.array_equal(s["wk"], w["wk"][:, heads.start * hs:heads.stop * hs])
        loc = local_shape(shape, tp, r)
        assert s["wq"].shape[1] == loc.head_num * hs and s["w2"].shape[2] == loc.hidden_dim
        # every local q head finds its kv head inside the rank's kv shard
        q_first = r * loc.head_num
        for h in range(loc.head_num):
            assert (q_first + h) // shape.kv_mul in heads
    if shape.group_size:
        from oracle.binding import Oracle
        o = Oracle()
        x = np.random.default_rng(0).standard_normal(shape.dim).astype(np.float32)
        full = o.matmul_w8(x, w["wo"][0], w["so"][0], shape.group_size)
        cols = shape.dim // tp
        part = sum(o.matmul_w8(x[r * cols:(r + 1) * cols], shards[r]["wo"][0], shards[r]["so"][0],
                               shape.group_size) for r in range(tp))
        assert np.abs(full - part).max() < 1e-4


def test_unshardable_shapes_are_refused():
    from kuiperllama_b200 import SHAPES, KllmError
    from kuiperllama_b200.tensor_parallel import check_shardable
    with pytest.raises(KllmError):
        check_shardable(SHAPES["small"], 2)          # 9 heads
    with pytest.raises(KllmError):
        check_shardable(SHAPES["tiny-int8"], 2)       # hidden 384: not a multiple of 256 int8 columns
    # int8 FFN shards: whole units of 256 columns, ranks may differ by one unit
    from kuiperllama_b200.tensor_parallel import ffn_range
    s7 = SHAPES["llama2-7b-int8"]
    assert [len(ffn_range(s7, 2, r)) for r in range(2)] == [5632, 5376]
    for tp in (2, 4, 8):
        check_shardable(s7, tp)
        cuts = [ffn_range(s7, tp, r) for r in range(tp)]
        assert cuts[0].start == 0 and cuts[-1].stop == s7.hidden_dim
        assert all(a.stop == b.start for a, b in zip(cuts, cuts[1:]))
        assert all(len(c) % 256 == 0 for c in cuts)
    check_shardable(SHAPES["tinyllama-1.1b"], 8)      # 4 kv heads replicated over 8 ranks
    check_shardable(SHAPES["llama2-7b"], 8)


def _gloo_rank(rank, world, key, steps, out_dir):
    import torch
    import torch.distributed as dist
    from kuiperllama_b200.tensor_parallel import local_shape, shard_weights
    from oracle.binding import Oracle
    shape, w = _full_model(key)
    shard = numpy_weights(shard_weights(shape, w, world, rank))

    def allreduce(v):
        t = torch.from_numpy(np.ascontiguousarray(v))
        dist.all_reduce(t)
        return t.numpy()

    m = OracleShardModel(Oracle(), shape, local_shape(shape, world, rank), shard, allreduce)
    tok, ids, logits = 1, [], None
    for pos in range(steps):
        tok, logits = m.step(tok, pos)
        ids.append(tok)
    np.savez(f"{out_dir}/rank{rank}.npz", ids=np.array(ids), logits=logits)


@pytest.mark.parametrize("key,world", [("small-tp", 2), ("small-tp", 4), ("small-tp", 8), ("small-int8", 2),
                                       ("small-tp-int8", 2), ("small-qwen", 2)])
def test_gloo_tensor_parallel_decode_matches_unsharded_oracle(oracle, tmp_path, key, world):
    from kuiperllama_b200.checkpoint import write_checkpoint
    steps = 12
    spawn(_gloo_rank, world, "gloo", (key, steps, str(tmp_path)))
    shape, w = _full_model(key)
    path = tmp_path / "full.bin"
    write_checkpoint(str(path), shape, w)
    om = oracle.open_model(path, shape.group_size > 0, shape.flavour)
    tok, ids = 1, []
    for pos in range(steps):
        tok, logits = om.step(tok, pos)
        ids.append(tok)
    om.close()
    for r in range(world):
        got = np.load(tmp_path / f"rank{r}.npz")
        assert list(got["ids"]) == ids, f"rank {r}"
        assert np.abs(got["logits"] - logits).max() < TOL
    # every rank holds the same residual stream -> the same logits, bit for bit
    a, b = np.load(tmp_path / "rank0.npz")["logits"], np.load(tmp_path / f"rank{world - 1}.npz")["logits"]
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


# ---- GPU: needs two devices ------------------------------------------------------------------

def _need_gpus(n):
    import torch
    if torch.cuda.device_count() < n:
        pytest.skip(f"needs {n} GPUs")


def _comm_rank(rank, world, backend, out_dir):
    import torch
    from kuiperllama_b200.tensor_parallel import Comm
    comm = Comm(4096, backend)
    g = torch.Generator(device="cuda").manual_seed(100 + rank)
    ok = True
    for batch in range(32):
        # 64 exchanges issued back to back (no host sync in between: the slot / sequence-flag
        # protocol has to keep fast and slow ranks apart on its own)
        sizes = [(4096, 2048, 256)[(batch + i) % 3] for i in range(64)]
        mine = [torch.empty(n, device="cuda").normal_(0, 1, generator=g) for n in sizes]
        res = [torch.full((n,), float(i), device="cuda") for i, n in enumerate(sizes)]
        want = []
        for i, n in enumerate(sizes):
            every = [torch.empty(n, device="cuda") for _ in range(world)]
            torch.distributed.all_gather(every, mine[i])
            total = every[0].clone()
            for r in range(1, world):  # rank-ordered fp32 adds: the kernel's order
                total += every[r]
            want.append(res[i] + total if i % 2 else total)
        torch.cuda.synchronize()
        got = [m.clone() for m in mine]
        for i in range(64):
            comm.allreduce_(got[i], residual=res[i] if i % 2 else None)
        torch.cuda.synchronize()
        if backend == "peer" or world == 2:  # rank-ordered by construction (a + b == b + a bitwise)
            ok = ok and all(bool(torch.equal(a, b)) for a, b in zip(got, want))
        else:  # NCCL picks its own reduction tree for more than two ranks
            ok = ok and all(bool(torch.allclose(a, b, rtol=1e-5, atol=1e-5)) for a, b in zip(got, want))
    comm.close()
    assert ok
    open(f"{out_dir}/ok{rank}", "w").write("1")


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["peer", "nccl"])
@pytest.mark.parametrize("world", [2, 4])
def test_comm_allreduce_matches_rank_ordered_sum(kllm_lib, tmp_path, backend, world):
    _need_gpus(world)
    spawn(_comm_rank, world, "nccl", (backend, str(tmp_path)))
    assert all((tmp_path / f"ok{r}").exists() for r in range(world))


def _decoder_rank(rank, world, key, backend, engine, steps, out_dir):
    import os
    os.environ["KLLM_ENGINE"] = engine
    import torch
    from kuiperllama_b200 import SHAPES, KllmError, synth_weights
    from kuiperllama_b200.tensor_parallel import Comm, comm_words, make_tp_decoder
    shape = SHAPES[key]
    full = synth_weights(shape, "cuda", 11)
    comm = Comm(comm_words(shape, world), backend)  # room for vocab / world words per rank
    try:
        dec = make_tp_decoder(shape, full, comm)
    except KllmError as e:
        # the persistent ring needs 16-byte weight/scale rows; forcing it on a shard it cannot
        # stage fails loudly (never a silent fallback) -- every rank sees the same refusal
        assert engine == "persistent" and "unsupported shape" in str(e), e
        open(f"{out_dir}/{backend}_{engine}_rank{rank}.refused", "w").write(str(e))
        comm.close()
        return
    assert dec.engine == engine
    # persistent engine: the classifier is sharded by vocabulary (each rank streams vocab / world rows and
    # publishes them to every rank); the graph engine keeps it replicated
    assert dec.classifier_rows == (shape.vocab_size // world if engine == "persistent" else shape.vocab_size)
    torch.distributed.barrier()  # the ranks' kernels wait for each other's partial sums: start together
    ids = dec.generate(1, 0, steps)
    logits = dec.logits()
    # the host-buffer path walks the same sequence
    tok, ids2 = 1, []
    for pos in range(8):
        tok = dec.step(tok, pos)
        ids2.append(tok)
    assert ids2 == ids[:8]
    np.savez(f"{out_dir}/{backend}_{engine}_rank{rank}.npz", ids=np.array(ids), logits=logits)
    dec.close()
    comm.close()


# transport x engine: the persistent megakernel exchanges tagged partials over peer memory itself;
# the graph engine calls the one-shot all-reduce kernel (peer) or ncclAllReduce
TP_MODES = [("peer", "persistent"), ("peer", "graph"), ("nccl", "graph")]


@pytest.mark.gpu
@pytest.mark.parametrize("key,world", [("small-tp", 2), ("small-int8", 2), ("small-tp-int8", 2), ("small-qwen", 2),
                                       ("small-tp", 4), ("small-tp", 8)])  # world 8: 8 heads / 2 kv heads -> kv heads replicated
def test_tp_decoder_matches_unsharded_oracle(kllm_lib, oracle, tmp_path, key, world):
    from kuiperllama_b200.checkpoint import write_checkpoint
    _need_gpus(world)
    steps = 48
    for backend, engine in TP_MODES:
        spawn(_decoder_rank, world, "nccl", (key, backend, engine, steps, str(tmp_path)))
    from kuiperllama_b200 import SHAPES, synth_weights
    shape = SHAPES[key]
    w = synth_weights(shape, "cuda", 11)
    path = tmp_path / "full.bin"
    write_checkpoint(str(path), shape, w)
    om = oracle.open_model(path, shape.group_size > 0, shape.flavour)
    tok, want = 1, []
    for pos in range(steps):
        tok, logits = om.step(tok, pos)
        want.append(tok)
    om.close()
    got = {}
    modes = [m for m in TP_MODES if not (tmp_path / f"{m[0]}_{m[1]}_rank0.refused").exists()]
    assert ("peer", "graph") in modes and ("nccl", "graph") in modes
    for backend, engine in modes:
        for r in range(world):
            g = np.load(tmp_path / f"{backend}_{engine}_rank{r}.npz")
            assert list(g["ids"]) == want, (backend, engine, r)
            assert np.abs(g["logits"] - logits).max() < TOL
            got[backend, engine, r] = g["logits"].view(np.uint32)
    # rank-ordered sums: every rank, and both peer-memory engines, hold identical bits
    ref = got["peer", "graph", 0]
    for r in range(world):
        assert np.array_equal(got["peer", "graph", r], ref)
        if ("peer", "persistent") in modes:
            assert np.array_equal(got["peer", "persistent", r], ref)
    if key in ("small-tp", "small-tp-int8", "small-qwen"):
        assert ("peer", "persistent") in modes, "the persistent engine must take this shape"


def _fast_rank(rank, world, key, steps, teacher, out_dir):
    import os
    os.environ["KLLM_ENGINE"] = "persistent"
    import torch
    from kuiperllama_b200 import SHAPES, synth_weights
    from kuiperllama_b200.tensor_parallel import Comm, make_tp_decoder
    shape = SHAPES[key]
    full = synth_weights(shape, "cuda", 11)
    comm = Comm(shape.dim, "peer")
    dec = make_tp_decoder(shape, full, comm, numerics="fast")
    assert dec.engine == "persistent"
    torch.distributed.barrier()
    logits = []
    for pos in range(steps):
        dec.step(teacher[pos], pos)
        logits.append(dec.logits())
    np.savez(f"{out_dir}/fast_rank{rank}.npz", logits=np.stack(logits))
    dec.close()
    comm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("key,world", [("small-tp", 2), ("small-tp-int8", 2), ("small-tp", 4)])
def test_tp_fast_numerics_within_tolerance_of_unsharded_exact(kllm_lib, tmp_path, key, world, monkeypatch):
    """Tensor parallel + numerics="fast" (flash-decoding attention over the rank's local heads, dp4a
    int8 rows): teacher-forced on the UNSHARDED exact decoder's tokens, every rank's logits stay within
    the north-star tolerance of the unsharded exact decoder at every position, and all ranks hold
    identical bits (rank-ordered sums)."""
    _need_gpus(world)
    from kuiperllama_b200 import SHAPES, Decoder, synth_weights
    monkeypatch.setenv("KLLM_ENGINE", "persistent")
    monkeypatch.setenv("KLLM_STAGE_BYTES", "8192")  # 32-timestep attention tiles: several tiles, several CTAs per head
    steps = 80
    shape = SHAPES[key]
    one = Decoder(shape, synth_weights(shape, "cuda", 11))
    tok, teacher, want = 1, [], []
    for pos in range(steps):
        teacher.append(tok)
        tok = one.step(tok, pos)
        want.append(one.logits())
    one.close()
    spawn(_fast_rank, world, "nccl", (key, steps, teacher, str(tmp_path)))
    got = [np.load(tmp_path / f"fast_rank{r}.npz")["logits"] for r in range(world)]
    worst = max(float(np.abs(got[0][pos] - want[pos]).max()) for pos in range(steps))
    assert 0.0 < worst <= TOL, worst
    for r in range(1, world):
        assert np.array_equal(got[r].view(np.uint32), got[0].view(np.uint32))
