"""-m gpu: the device-resident decoder (kllm_decoder_*) against
  - the reference PyTorch logits committed under tests/golden (<= 1e-4, north-star tolerance),
  - the CPU oracle (same tolerance, identical greedy ids),
  - the reference's OWN CUDA model path run on this GPU (oracle/_ref): bit-identical logits,
    KV cache and token ids -- including at BASELINE.json's full TinyLlama-1.1B size; live when
    oracle/_ref is built, and always against its recorded outputs (tests/reference_outputs.py)."""
import ctypes
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from gpu_util import assert_bit_equal, sync
from reference_outputs import check, live_reference

pytestmark = pytest.mark.gpu

TOL = 1e-4  # BASELINE.json north_star: logits within 1e-4 fp32


@pytest.fixture(autouse=True, params=["persistent", "graph"])
def engine(request, monkeypatch):
    """Every decoder test runs on both engines: the persistent megakernel (TMA weight ring, one
    cooperative launch) and the CUDA-graph chain of fused launches."""
    monkeypatch.setenv("KLLM_ENGINE", request.param)
    return request.param


def make_decoder(shape, w):
    """Decoder on the engine the `engine` fixture forces.  The persistent ring needs 16-byte
    weight/scale rows; forcing it on a shape it cannot stage must fail loudly (never silently
    fall back) -- such cases are skipped here and covered by the graph engine run."""
    from kuiperllama_b200 import Decoder, KllmError
    try:
        return Decoder(shape, w)
    except KllmError as e:
        if os.environ.get("KLLM_ENGINE") == "persistent" and "unsupported shape" in str(e):
            pytest.skip(f"{shape.name}: persistent engine refuses this shape (graph engine covers it)")
        raise


def load_decoder(path, quant=False, flavour="llama2", qkv_bias=None):
    from kuiperllama_b200.checkpoint import read_checkpoint, to_device
    shape, w = read_checkpoint(str(path), quant, flavour, qkv_bias=qkv_bias)
    return make_decoder(shape, to_device(w)), shape


@pytest.fixture(scope="module")
def ref():
    return live_reference("llama2")


class RefModel:
    def __init__(self, ref, path, quant, vocab):
        self.L = ref.L
        self.h = self.L.kref_model_create(str(path).encode(), int(quant))
        assert self.h, "reference LLama2Model::init failed"
        self.vocab = vocab
        self.buf = np.empty(vocab, np.float32)

    def step(self, token, pos, want_logits=True):
        p = self.buf.ctypes.data_as(ctypes.POINTER(ctypes.c_float)) if want_logits else None
        nxt = self.L.kref_model_step(self.h, int(token), int(pos), p, self.vocab)
        return nxt, (self.buf.copy() if want_logits else None)

    def close(self):
        self.L.kref_model_destroy(self.h)


GOLDENS = [("tiny_llama2_fp32_shared", False, "llama2", None), ("tiny_llama2_fp32", False, "llama2", None),
           ("tiny_llama2_int8", True, "llama2", None), ("tiny_qwen2file_fp32", False, "llama2", True)]


@pytest.mark.parametrize("name,quant,flavour,bias", GOLDENS)
def test_golden_logits(kllm_lib, oracle, name, quant, flavour, bias):
    g = np.load(GOLDEN / f"{name}.npz")
    dec, shape = load_decoder(GOLDEN / f"{name}.bin", quant, flavour, bias)
    om = oracle.open_model(GOLDEN / f"{name}.bin", quant, "qwen2file" if bias else flavour)
    for t, tok in enumerate(g["tokens"]):
        nxt = dec.step(int(tok), t)
        logits = dec.logits()
        o_next, o_logits = om.step(int(tok), t)
        assert np.abs(logits - g["logits"][t]).max() < TOL, (name, t)
        assert np.abs(logits - o_logits).max() < TOL
        assert nxt == int(np.argmax(g["logits"][t])) == o_next
    k, v = dec.kv_cache(); ok, ov = om.kv_cache()
    n = len(g["tokens"])
    assert np.abs(k[:, :n] - ok[:, :n]).max() < TOL
    assert np.abs(v[:, :n] - ov[:, :n]).max() < TOL
    om.close(); dec.close()


@pytest.mark.parametrize("name,quant", [("tiny_llama2_fp32_shared", False), ("tiny_llama2_fp32", False),
                                        ("tiny_llama2_int8", True)])
def test_bit_exact_vs_reference_cuda_model_goldens(kllm_lib, ref, name, quant):
    g = np.load(GOLDEN / f"{name}.npz")
    dec, shape = load_decoder(GOLDEN / f"{name}.bin", quant)
    rm = RefModel(ref, GOLDEN / f"{name}.bin", quant, shape.vocab_size) if ref else None
    ids, logits, r_ids, r_logits = [], [], [], []
    for t, tok in enumerate(g["tokens"]):
        ids.append(dec.step(int(tok), t))
        logits.append(dec.logits())
        if rm:
            r_next, r_lg = rm.step(int(tok), t)
            r_ids.append(r_next); r_logits.append(r_lg)
    check(logits, r_logits if rm else None, f"model/{name}/logits", f"{name} logits [position, vocab]")
    check(ids, r_ids if rm else None, f"model/{name}/ids", f"{name} token ids")
    if rm:
        rm.close()
    dec.close()


def _reference_free_run(ref, path, shape, steps):
    """Greedy ids of `steps` free-running positions from token 1 and the last position's logits on the
    reference's CUDA path (demo/main.cpp loop); (None, None) without a reference build."""
    if not ref:
        return None, None
    rm = RefModel(ref, path, shape.group_size > 0, shape.vocab_size)
    tok, ids = 1, []
    for pos in range(steps):
        tok, lg = rm.step(tok, pos, want_logits=(pos == steps - 1))
        ids.append(tok)
    rm.close()
    return ids, lg


def _synth_file(tmp_path, key, seed):
    from kuiperllama_b200 import SHAPES, synth_weights
    from kuiperllama_b200.checkpoint import write_checkpoint
    shape = SHAPES[key]
    w = synth_weights(shape, "cuda", seed)
    path = tmp_path / f"{key}.bin"
    write_checkpoint(str(path), shape, w)
    return shape, w, path


@pytest.mark.parametrize("key,steps", [("tiny", 64), ("tiny-shared", 64), ("small", 160), ("small-hs48", 160),
                                       ("tiny-int8", 64), ("small-int8", 96)])
def test_free_running_decode_identical_to_reference_cuda(kllm_lib, ref, tmp_path, key, steps):
    """Greedy decode feeding its own output: token ids AND final logits identical to the
    reference's CUDA path (demo/main.cpp loop), every position up to seq_len."""
    from kuiperllama_b200 import Decoder
    shape, w, path = _synth_file(tmp_path, key, 100 + steps)
    dec = make_decoder(shape, w)
    mine = dec.generate(1, 0, steps)
    theirs, lg = _reference_free_run(ref, path, shape, steps)
    check(mine, theirs, f"free_run/{key}/{steps}/ids", f"{key}: token ids of {steps} free-running steps")
    check(dec.logits(), lg, f"free_run/{key}/{steps}/logits", f"{key}: logits after {steps} free-running steps")
    # the host-buffer path (predict semantics) walks the same sequence
    tok = 1
    for pos in range(8):
        tok = dec.step(tok, pos)
        assert tok == mine[pos]
    assert dec.step(5, 3, is_prompt=True) == -1  # predict(..., is_prompt=true) returns -1
    dec.close()


@pytest.mark.parametrize("qkey", ["tiny-qwen", "small-qwen"])
def test_qwen2_flavour_vs_cpu_oracle(kllm_lib, oracle, tmp_path, qkey):
    """QWEN2_SUPPORT arithmetic (half-split RoPE, theta 1e6, eps 1e-6, qkv bias, GQA kv_mul 2):
    no reference CUDA *model* build exists for this flavour (its tokenizer needs absl/re2), so
    the whole-model check is against the CPU oracle; the kernels themselves are bit-checked
    against the reference's QWEN2 kernels in test_kernels_gpu.py."""
    from kuiperllama_b200 import Decoder
    shape, w, path = _synth_file(tmp_path, qkey, 7)
    dec = make_decoder(shape, w)
    om = oracle.open_model(path, False, "qwen2")
    tok = 1
    for pos in range(48):
        nxt = dec.step(tok, pos)
        o_next, o_logits = om.step(tok, pos)
        lg = dec.logits()
        assert np.abs(lg - o_logits).max() < TOL, pos
        top2 = np.sort(o_logits)[-2:]
        if top2[1] - top2[0] > 2 * TOL:
            assert nxt == o_next, pos
        tok = o_next
    om.close(); dec.close()


def test_teacher_forced_generate_and_determinism(kllm_lib, engine):
    from kuiperllama_b200 import SHAPES, Decoder, synth_weights
    shape = SHAPES["small"]
    dec = make_decoder(shape, synth_weights(shape, "cuda", 11))
    free = dec.generate(1, 0, 100)
    again = dec.generate(1, 0, 100)
    assert free == again  # bitwise deterministic
    inputs = [1] + free[:-1]
    forced = dec.generate(0, 0, 100, teacher=inputs)
    assert forced == free
    assert dec.engine == engine
    assert dec.launches_per_step == (1 if engine == "persistent" else 6 * shape.layer_num + 3)
    dec.close()


def test_tinyllama_full_size_identical_to_reference_cuda(kllm_lib, ref, tmp_path, engine):
    """BASELINE.json config 2 at full size (dim 2048, 22 layers, 32/4 heads, vocab 32000):
    256 free-running greedy steps; ids, final logits and the KV cache must be identical to the
    reference's own CUDA path.  Then determinism over the full 1024-token run."""
    from kuiperllama_b200 import SHAPES, Decoder, synth_weights
    from kuiperllama_b200.checkpoint import write_checkpoint
    shape = SHAPES["tinyllama-1.1b"]
    w = synth_weights(shape, "cuda", 1235)
    ckpt_dir = "/dev/shm" if os.path.isdir("/dev/shm") else str(tmp_path)
    path = os.path.join(ckpt_dir, "kllm_tinyllama_test.bin")
    try:
        write_checkpoint(path, shape, w)
        dec = make_decoder(shape, w)
        assert dec.engine == engine
        steps = 256
        mine = dec.generate(1, 0, steps)
        theirs, lg = _reference_free_run(ref, path, shape, steps)
        check(mine, theirs, "free_run/tinyllama-1.1b/256/ids", "TinyLlama-1.1B token ids of 256 steps")
        check(dec.logits(), lg, "free_run/tinyllama-1.1b/256/logits", "TinyLlama-1.1B logits after 256 steps")
    finally:
        if os.path.exists(path):
            os.remove(path)
    full = dec.generate(1, 0, 1024)
    assert full[:steps] == mine
    assert dec.generate(1, 0, 1024) == full
    dec.close()


def test_default_engine_selection(kllm_lib, monkeypatch):
    """Without KLLM_ENGINE the decoder picks the persistent megakernel when the shape fits its
    ring and the graph engine otherwise -- both CUDA, never a CPU path."""
    from kuiperllama_b200 import SHAPES, Decoder, synth_weights
    monkeypatch.delenv("KLLM_ENGINE", raising=False)
    for key, want in (("small", "persistent"), ("small-int8", "persistent"), ("tiny-int8", "graph")):
        shape = SHAPES[key]
        dec = Decoder(shape, synth_weights(shape, "cuda", 3))
        assert dec.engine == want, key
        dec.close()
    from kuiperllama_b200.checkpoint import read_checkpoint, to_device
    shape, w = read_checkpoint(str(GOLDEN / "tiny_llama2_int8.bin"), True)
    dec = Decoder(shape, to_device(w))  # 4-byte scale rows: not bulk-copyable
    assert dec.engine == "graph"
    dec.close()


RING_STRESS = {
    # many ring stages per phase / several ring revolutions per phase / MHA with 32 kv heads:
    # dim, hidden, layers, heads, kv_heads, vocab, seq_len   (regressions: mbarrier phase aliasing)
    "dim2048_hid5632": (2048, 5632, 1, 32, 4, 1024, 64),
    "dim2048_vocab32000": (2048, 2048, 1, 32, 4, 32000, 64),
    "dim2048_mha32": (2048, 2048, 1, 32, 32, 1024, 64),
    "dim1024_hid5632": (1024, 5632, 2, 16, 4, 1024, 64),
}


@pytest.mark.parametrize("name", sorted(RING_STRESS))
def test_persistent_equals_graph_on_ring_stress_shapes(kllm_lib, monkeypatch, name):
    """The graph engine is checked bit for bit against the reference CUDA path above; here the
    persistent megakernel must reproduce it (ids and logits) on shapes that drive the stage ring
    through many revolutions per phase."""
    from kuiperllama_b200 import Decoder, ModelShape, synth_weights
    d, h, L, nh, nkv, V, S = RING_STRESS[name]
    shape = ModelShape(name, d, h, L, nh, nkv, V, S)
    w = synth_weights(shape, "cuda", 5)
    monkeypatch.setenv("KLLM_ENGINE", "graph")
    a = Decoder(shape, w)
    ids_a = a.generate(1, 0, 48)
    la = a.logits()
    a.close()
    monkeypatch.setenv("KLLM_ENGINE", "persistent")
    b = Decoder(shape, w)
    ids_b = b.generate(1, 0, 48)
    assert ids_a == ids_b
    assert_bit_equal(la, b.logits(), name)
    b.close()


# ---- BASELINE.json configs[2] and configs[3] at FULL size ------------------------------------------
_FULL_CACHE = {}


def _full_size_case(key, seed):
    """Weights + checkpoint file of a full-size workload, built once per test session (both engine
    parametrisations reuse it).  The file lives in /dev/shm: the reference mmaps it."""
    if key not in _FULL_CACHE:
        from kuiperllama_b200 import SHAPES, synth_weights
        from kuiperllama_b200.checkpoint import write_checkpoint
        shape = SHAPES[key]
        w = synth_weights(shape, "cuda", seed)
        path = os.path.join("/dev/shm" if os.path.isdir("/dev/shm") else "/tmp", f"kllm_full_{key}.bin")
        write_checkpoint(path, shape, w)
        _FULL_CACHE[key] = {"shape": shape, "w": w, "path": path}
    return _FULL_CACHE[key]


@pytest.fixture(scope="module", autouse=True)
def _drop_full_size_files():
    yield
    for case in _FULL_CACHE.values():
        if os.path.exists(case["path"]):
            os.remove(case["path"])
    _FULL_CACHE.clear()


def test_llama2_7b_int8_full_size_identical_to_reference_cuda(kllm_lib, ref, engine):
    """BASELINE.json configs[2] at full size (dim 4096, 32 layers, MHA 32/32, hidden 11008, vocab
    32000, int8 group 64 as export.py --version 3 writes it): 128 free-running greedy steps -- token
    ids AND the final logits bit-identical to the reference's own CUDA path loading the same file
    (llama3.cpp:184-288, matmul_kernel.cu:56-87)."""
    case = _full_size_case("llama2-7b-int8", 1236)
    shape = case["shape"]
    steps = 128
    if "ref_ids" not in case:
        case["ref_ids"], case["ref_logits"] = _reference_free_run(ref, case["path"], shape, steps)
    dec = make_decoder(shape, case["w"])
    assert dec.engine == engine
    mine = dec.generate(1, 0, steps)
    check(mine, case["ref_ids"], "free_run/llama2-7b-int8/128/ids", "Llama-2-7B int8 token ids of 128 steps")
    check(dec.logits(), case["ref_logits"], "free_run/llama2-7b-int8/128/logits", "Llama-2-7B int8 logits after 128 steps")
    # host-buffer path (predict semantics) at a late position reproduces the same id
    assert dec.step(mine[steps - 2], steps - 1) == mine[steps - 1]
    dec.close()


def test_qwen25_05b_full_size(kllm_lib, oracle, engine):
    """BASELINE.json configs[3] at full size (dim 896, 24 layers, GQA 14/2 -> kv_mul 7, hidden 4864,
    vocab 151936 shared classifier, seq_len 32768, qkv bias, half-split RoPE theta 1e6, eps 1e-6).
    No reference CUDA *model* build exists for the QWEN2 flavour here (its tokenizer needs
    absl/re2), so the whole-model check is the CPU oracle, teacher-forced, north-star tolerance:
    logits within 1e-4 and the same greedy id wherever the top-2 margin exceeds 2e-4.  Both engines
    must then agree with EACH OTHER bit for bit over a long free-running decode (context 1 -> 1100),
    which carries the graph engine's kernel-level bit-exactness (test_kernels_gpu.py, QWEN2 kernels)
    to the persistent megakernel at kv_mul 7."""
    case = _full_size_case("qwen2.5-0.5b", 1237)
    shape = case["shape"]
    dec = make_decoder(shape, case["w"])
    assert dec.engine == engine
    n_oracle = 20
    if "oracle" not in case:
        om = oracle.open_model(case["path"], False, "qwen2")
        tok, rows = 1, []
        for pos in range(n_oracle):
            nxt, lg = om.step(tok, pos)
            rows.append((tok, nxt, lg.copy()))
            tok = nxt
        om.close()
        case["oracle"] = rows
    for pos, (tok, o_next, o_logits) in enumerate(case["oracle"]):
        nxt = dec.step(tok, pos)
        lg = dec.logits()
        assert np.abs(lg - o_logits).max() < TOL, pos
        top2 = np.sort(o_logits)[-2:]
        if top2[1] - top2[0] > 2 * TOL:
            assert nxt == o_next, pos
    steps = 1100
    ids = dec.generate(1, 0, steps)
    lg = dec.logits()
    if "free" in case:
        other_engine, other_ids, other_lg = case["free"]
        assert other_engine != engine
        assert ids == other_ids, f"{engine} and {other_engine} engines diverge on Qwen2.5-0.5B"
        assert_bit_equal(lg, other_lg, "Qwen2.5-0.5B logits after 1100 free-running steps, engine vs engine")
    else:
        case["free"] = (engine, ids, lg)
    dec.close()


@pytest.mark.parametrize("key", ["small", "small-int8", "small-qwen"])
def test_prompt_call_equals_stepping(kllm_lib, key):
    """kllm_decoder_prompt (one launch, classifier skipped for all but the last prompt position --
    llama3.cpp:738-739 throws those logits away) leaves the same KV cache, logits and next id as
    predict()-style stepping with is_prompt = true, bit for bit, and decoding continues identically."""
    from kuiperllama_b200 import SHAPES, synth_weights
    shape = SHAPES[key]
    w = synth_weights(shape, "cuda", 21)
    rng = np.random.default_rng(5)
    toks = [1] + [int(t) for t in rng.integers(2, shape.vocab_size, 37)]
    a = make_decoder(shape, w)
    nxt_a = a.prompt(toks)
    ka, va = a.kv_cache()
    la = a.logits()
    b = make_decoder(shape, w)
    nb = -2
    for pos, t in enumerate(toks):
        nb = b.step(t, pos, is_prompt=(pos < len(toks) - 1))
        assert (nb == -1) == (pos < len(toks) - 1)
    kb, vb = b.kv_cache()
    n = len(toks)
    assert nxt_a == nb
    assert_bit_equal(ka[:, :n], kb[:, :n], "key cache after the prompt")
    assert_bit_equal(va[:, :n], vb[:, :n], "value cache after the prompt")
    assert_bit_equal(la, b.logits(), "logits of the last prompt position")
    assert a.generate(nxt_a, n, 24) == b.generate(nb, n, 24)
    a.close(); b.close()


@pytest.mark.parametrize("key,steps,stage_bytes", [
    ("small-int8", 64, None), ("small-tp-int8", 64, None), ("small-int8", 90, 8192),
    ("small", 150, 4096),        # fp32, head_size 32: 32-timestep tiles -> 5 tiles over 4 CTAs per head
    ("small-qwen", 120, 8192),   # qwen RoPE pairing, q/k/v biases; 32-timestep tiles, one CTA per head
    ("tinyllama-1.1b", 700, None),  # BASELINE.json configs[1]: 128-timestep tiles, GQA 8:1
    ("llama2-7b-int8", 200, None)])  # configs[2]: dp4a rows + 32-timestep tiles, 16 threads per timestep
def test_fast_numerics_within_north_star_tolerance(kllm_lib, monkeypatch, key, steps, stage_bytes):
    """numerics="fast" (persistent engine): int8 rows as 24-bit fixed-point activations x int8 weights
    on dp4a, attention as flash-decoding (split by timestep over several CTAs per head, online softmax,
    partials merged).  TOLERANCED against the bit-exact mode (which the tests above pin to the
    reference's CUDA path): teacher-forced on the exact mode's tokens, logits within 1e-4 (north-star
    tolerance) at every position and the same greedy id wherever the exact top-2 margin exceeds 2e-4."""
    from kuiperllama_b200 import SHAPES, Decoder, synth_weights
    monkeypatch.setenv("KLLM_ENGINE", "persistent")
    if stage_bytes:
        monkeypatch.setenv("KLLM_STAGE_BYTES", str(stage_bytes))
    if key in _FULL_CACHE or key == "llama2-7b-int8":
        case = _full_size_case(key, 1236)
        shape, w = case["shape"], case["w"]
    else:
        shape = SHAPES[key]
        w = synth_weights(shape, "cuda", 31)
    exact = Decoder(shape, w)
    fast = Decoder(shape, w, numerics="fast")
    assert exact.engine == fast.engine == "persistent"
    tok, worst, checked = 1, 0.0, 0
    for pos in range(steps):
        a = exact.step(tok, pos)
        b = fast.step(tok, pos)
        la, lb = exact.logits(), fast.logits()
        worst = max(worst, float(np.abs(la - lb).max()))
        top2 = np.sort(la)[-2:]
        if top2[1] - top2[0] > 2 * TOL:
            assert a == b, pos
            checked += 1
        tok = a
    assert worst <= TOL, worst
    assert worst > 0.0, "the fast mode produced bit-identical logits: it did not run"
    # free-running determinism of the fast mode
    assert fast.generate(1, 0, 32) == fast.generate(1, 0, 32)
    exact.close(); fast.close()


@pytest.mark.parametrize("key,steps,warps", [("small-int8", 64, None), ("small-tp-int8", 64, "12"),
                                             ("llama2-7b-int8", 48, None), ("llama2-7b-int8", 48, "12")])
def test_int8_tensor_core_team_form_within_tolerance(kllm_lib, monkeypatch, key, steps, warps):
    """KLLM_INT8_MMA=1 (opt-in): int8 fast rows in the team form -- stages of 3-8 rows through mma.sync m16n8k32
    s8 (weight rows x the three digit planes of x), one or two long rows on dp4a with the columns split over the
    team; pairs of warps (14 consumer warps) or teams of four (12).  Same fixed-point arithmetic as the default
    dp4a rows, different float summation order: TOLERANCED against the exact mode like the default fast mode."""
    from kuiperllama_b200 import SHAPES, Decoder, synth_weights
    monkeypatch.setenv("KLLM_ENGINE", "persistent")
    if key == "llama2-7b-int8":
        case = _full_size_case(key, 1236)
        shape, w = case["shape"], case["w"]
    else:
        shape = SHAPES[key]
        w = synth_weights(shape, "cuda", 31)
    exact = Decoder(shape, w)
    monkeypatch.setenv("KLLM_INT8_MMA", "1")
    if warps:
        monkeypatch.setenv("KLLM_CONSUMER_WARPS", warps)
    team = Decoder(shape, w, numerics="fast")
    monkeypatch.delenv("KLLM_INT8_MMA")
    monkeypatch.delenv("KLLM_CONSUMER_WARPS", raising=False)
    plain = Decoder(shape, w, numerics="fast")
    tok, worst, differs = 1, 0.0, False
    for pos in range(steps):
        a = exact.step(tok, pos)
        b = team.step(tok, pos)
        plain.step(tok, pos)
        la, lb = exact.logits(), team.logits()
        worst = max(worst, float(np.abs(la - lb).max()))
        differs = differs or not np.array_equal(lb, plain.logits())
        top2 = np.sort(la)[-2:]
        if top2[1] - top2[0] > 2 * TOL:
            assert a == b, pos
        tok = a
    assert worst <= TOL, worst
    assert differs, "the team form produced the plain dp4a rows' bits: it did not run"
    for d in (exact, team, plain):
        d.close()


def test_fast_numerics_by_environment(kllm_lib, monkeypatch):
    """KLLM_MODE=fast overrides the descriptor's numerics at create time (and KLLM_MODE=exact a
    descriptor that asks for fast)."""
    from kuiperllama_b200 import SHAPES, Decoder, synth_weights
    monkeypatch.setenv("KLLM_ENGINE", "persistent")
    shape = SHAPES["small-int8"]
    w = synth_weights(shape, "cuda", 31)
    exact = Decoder(shape, w)
    monkeypatch.setenv("KLLM_MODE", "fast")
    by_env = Decoder(shape, w)
    monkeypatch.setenv("KLLM_MODE", "exact")
    forced_exact = Decoder(shape, w, numerics="fast")
    monkeypatch.delenv("KLLM_MODE")
    by_desc = Decoder(shape, w, numerics="fast")
    for pos in range(40):
        t = exact.step(1 + pos, pos)
        for d in (by_env, forced_exact, by_desc):
            d.step(1 + pos, pos)
    assert_bit_equal(exact.logits(), forced_exact.logits(), "KLLM_MODE=exact")
    assert_bit_equal(by_env.logits(), by_desc.logits(), "KLLM_MODE=fast vs numerics=fast")
    assert not np.array_equal(exact.logits(), by_env.logits())
    for d in (exact, by_env, forced_exact, by_desc):
        d.close()
