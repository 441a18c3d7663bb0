"""-m gpu: batched int8 prompt prefill on tcgen05.mma.kind::i8 (kllm_gemm_w8, kllm_decoder_prefill_w8).

kllm_gemm_w8 computes out[T, N] = x[T, K] . (s (.) w)[N, K]^T with x turned, per token and 64-group g, into
step_g * q (step_g = gmax_g * 2^-22, q = rint(x * 2^22 / gmax_g), three balanced int8 digit planes).

Stated bounds, derived:
  * Integer path.  E = sum_g s_g step_g Q_g with Q_g = sum_i w_i q_i is formed here in float64 from the same
    quantised x (exact: |Q_g| <= 2^35, every product and partial sum an integer below 2^53).  The device gets
    the three digit dot products D_k exactly (int32 on the tensor cores) and rounds three times per group --
    fma(D1, 256, D0), fma(D2, 65536, .), step * s -- then accumulates G = K / 64 terms with fma.  So
        |out - E| <= (G + 4) * 2^-24 * B,   B = sum_g |s_g step_g| (65536 |D2| + 256 |D1| + |D0|)
    and B <= (|step| * (65536|a2| + 256|a1| + |a0|)) . (|s| |w|)^T, which is what is evaluated.  A wrong
    field in the instruction descriptor (signedness, D type) or a lost digit plane is off by far more.
  * Quantisation.  |x_i - step q_i| <= step / 2 = 2^-23 gmax_g, so against the float64 product of x and the
    dequantised weights the error stays within the bound above plus sum_i 2^-23 gmax_g(i) |s w_i|.
  * Decoder.  kllm_decoder_prefill_w8 against the bit-exact position-by-position prompt() on the same engine:
    logits within 1e-4 (the north-star tolerance), the same greedy id wherever the exact top-2 margin exceeds
    2e-4, K / V rows within 1e-4 * (row rms + 1e-3), and 16 teacher-forced decode steps from the prefilled
    cache within 1e-4.  Only x is rounded, to 2^-23 of its group maximum -- the fp32 level -- so these are
    the fast decode mode's bounds (test_decoder_gpu.py)."""
import ctypes
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from gpu_util import ptr, sync

pytestmark = pytest.mark.gpu

TOL = 1e-4


def workspace_bytes(T, K):
    return 3 * T * K + 4 * (K // 64) * ((T + 63) // 64 * 64)


def quantise_x(x):
    """The device quantiser (kllm_device.cuh w8_group_step / w8_group_inv / w8_digits4) in fp32 torch:
    returns step [T, G] fp32, q [T, K] int64 and the digit planes a0, a1, a2 [T, K] int64."""
    T, K = x.shape
    xg = x.view(T, K // 64, 64)
    gmax = xg.abs().amax(dim=2)
    step = gmax * torch.tensor(2.0 ** -22, dtype=torch.float32, device=x.device)
    inv = torch.where(gmax > 0, torch.tensor(4194304.0, device=x.device) / gmax, torch.zeros_like(gmax))
    q = torch.round(xg * inv[:, :, None]).to(torch.int64).view(T, K)  # fp32 product, round half to even
    a0 = ((q + 128) & 255) - 128
    q1 = (q - a0) >> 8
    a1 = ((q1 + 128) & 255) - 128
    a2 = (q1 - a1) >> 8
    assert torch.equal(65536 * a2 + 256 * a1 + a0, q)
    assert int(torch.stack([a0, a1, a2]).abs().max()) <= 128
    return step, q, a0, a1, a2


def make_inputs(T, K, N, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    G = K // 64
    x = torch.empty(T, K, device="cuda").normal_(0, 1, generator=g)
    # mixed-magnitude groups: group g scaled by 10^((g % 7) - 3)
    mag = torch.tensor([10.0 ** ((i % 7) - 3) for i in range(G)], device="cuda")
    x = (x.view(T, G, 64) * mag[None, :, None]).view(T, K).contiguous()
    if G > 1:
        x[:, 1 * 64:2 * 64] = 0  # an all-zero group (step 0) for every token
    x[0, :64] = 0                # and one for token 0 alone
    w = torch.randint(-127, 128, (N, K), device="cuda", generator=g, dtype=torch.int64)
    w[:, :8] = 127               # weights at the ends of the int8 range
    w[::3, 8:16] = -128
    w = w.to(torch.int8).contiguous()
    s = (torch.rand(N, G, device="cuda", generator=g) + 0.5) * (0.02 / 127)
    return x, w, s.contiguous()


def run_gemm(lib, x, w, s, T, K, N):
    ws = torch.empty(workspace_bytes(T, K), dtype=torch.uint8, device="cuda")
    out = torch.full((T, N), float("nan"), device="cuda")
    rc = lib.kllm_gemm_w8(ptr(x), ptr(w), ptr(s), ptr(out), ptr(ws), T, K, N, None)
    assert rc == 0, rc
    sync()
    return out


SHAPES = [
    # T, K, N: every T in {1, 7, 64, 65, 200, 256, 300}, K in {64, 128, 384, 4096, 11008},
    # N in {96, 128, 1000, 4096, 11008}; the Llama-2-7B projection shapes at T = 256 and 300
    (1, 64, 96), (7, 128, 128), (64, 384, 1000), (65, 64, 11008), (1, 11008, 128), (7, 4096, 1000),
    (200, 64, 96), (256, 128, 4096), (300, 384, 96), (65, 4096, 4096), (200, 11008, 4096),
    (256, 4096, 11008), (300, 11008, 1000), (256, 11008, 4096), (300, 4096, 4096), (64, 11008, 11008),
]


@pytest.mark.parametrize("T,K,N", SHAPES)
def test_gemm_w8_integer_path_exact(kllm_lib, T, K, N):
    x, w, s = make_inputs(T, K, N, T * 131 + K * 7 + N)
    out = run_gemm(kllm_lib, x, w, s, T, K, N)
    assert torch.isfinite(out).all()
    G = K // 64
    step, q, a0, a1, a2 = quantise_x(x)
    stepk = step.double().repeat_interleave(64, dim=1)  # [T, K]
    wd = (w.double().view(N, G, 64) * s.double()[:, :, None]).view(N, K)
    exact = (stepk * q.double()) @ wd.t()  # sum_g s_g step_g Q_g, exact in float64
    mag = stepk * (65536 * a2.abs() + 256 * a1.abs() + a0.abs()).double()
    bound = (G + 4) * 2.0 ** -24 * (mag @ wd.abs().t()) + 1e-30
    err = (out.double() - exact).abs()
    assert bool((err <= bound).all()), f"max err/bound {float((err / bound).max()):.3f}"
    # against the unquantised activations: + the quantisation step of every element
    full = x.double() @ wd.t()
    qbound = bound + (2.0 ** -23 * (step.double() * 4194304.0).repeat_interleave(64, dim=1)) @ wd.abs().t()
    qerr = (out.double() - full).abs()
    assert bool((qerr <= qbound).all()), f"max err/bound {float((qerr / qbound).max()):.3f}"
    print(f"[gemm_w8] T={T} K={K} N={N}: max err/bound {float((err / bound).max()):.3e}, "
          f"vs unquantised max rel {float(qerr.max() / full.abs().max().clamp_min(1e-30)):.3e}")


def test_gemm_w8_rejects_before_launch(kllm_lib):
    T, K, N = 4, 128, 8
    x = torch.zeros(T, K + 4, device="cuda")
    w = torch.zeros(N, K + 64, dtype=torch.int8, device="cuda")
    s = torch.ones(N, 4, device="cuda")
    out = torch.zeros(T, N, device="cuda")
    ws = torch.zeros(workspace_bytes(T, K + 64) + 64, dtype=torch.uint8, device="cuda")
    sync()
    before = kllm_lib.kllm_launch_count()
    f = kllm_lib.kllm_gemm_w8
    assert f(ptr(x), ptr(w), ptr(s), ptr(out), ptr(ws), T, 96, N, None) == -2   # K % 64 != 0
    assert f(ptr(x), ptr(w), ptr(s), ptr(out), ptr(ws), T, 100, N, None) == -2
    assert f(None, ptr(w), ptr(s), ptr(out), ptr(ws), T, K, N, None) == -1
    assert f(ptr(x), None, ptr(s), ptr(out), ptr(ws), T, K, N, None) == -1
    assert f(ptr(x), ptr(w), None, ptr(out), ptr(ws), T, K, N, None) == -1
    assert f(ptr(x), ptr(w), ptr(s), None, ptr(ws), T, K, N, None) == -1
    assert f(ptr(x), ptr(w), ptr(s), ptr(out), None, T, K, N, None) == -1
    assert f(ptr(x), ptr(w), ptr(s), ptr(out), ptr(ws), 0, K, N, None) == -1
    assert f(ptr(x), ptr(w), ptr(s), ptr(out), ptr(ws), T, K, 0, None) == -1
    off = lambda t, n: ctypes.c_void_p(t.data_ptr() + n)  # noqa: E731
    assert f(off(x, 4), ptr(w), ptr(s), ptr(out), ptr(ws), T, K, N, None) == -2   # unaligned bases
    assert f(ptr(x), off(w, 8), ptr(s), ptr(out), ptr(ws), T, K, N, None) == -2
    assert f(ptr(x), ptr(w), ptr(s), ptr(out), off(ws, 8), T, K, N, None) == -2
    assert f(ptr(x), ptr(w), off(s, 2), ptr(out), ptr(ws), T, K, N, None) == -2
    assert f(ptr(x), ptr(w), ptr(s), off(out, 2), ptr(ws), T, K, N, None) == -2
    assert kllm_lib.kllm_launch_count() == before, "a refused call launched a kernel"


def _decoder(shape, w):
    from kuiperllama_b200 import Decoder, KllmError
    try:
        return Decoder(shape, w)
    except KllmError as e:
        if os.environ.get("KLLM_ENGINE") == "persistent" and "unsupported shape" in str(e):
            pytest.skip(f"{shape.name}: the persistent engine refuses this shape (the graph engine run covers it)")
        raise


def _rows_close(a, b, n):
    worst = 0.0
    for x, y in zip(a, b):
        x, y = x[:, :n].astype(np.float64), y[:, :n].astype(np.float64)
        rms = np.sqrt((x ** 2).mean(axis=-1, keepdims=True))
        worst = max(worst, float((np.abs(x - y) / (rms + 1e-3)).max()))
    return worst


CASES = [("small-int8", 70, 0), ("small-int8", 70, 29), ("tiny-int8", 40, 0), ("small-tp-int8", 80, 0),
         ("llama2-7b-int8", 300, 0), ("llama2-7b-int8", 300, 100)]


@pytest.mark.parametrize("engine", ["persistent", "graph"])
@pytest.mark.parametrize("key,n_prompt,split", CASES)
def test_prefill_w8_matches_prompt(kllm_lib, monkeypatch, engine, key, n_prompt, split):
    """prefill_w8 (after prompt() for the first `split` tokens when split > 0) against prompt() of the whole
    prompt on the same weights and engine; then 16 teacher-forced decode steps from both caches."""
    from kuiperllama_b200 import SHAPES, synth_weights
    monkeypatch.setenv("KLLM_ENGINE", engine)
    shape = SHAPES[key]
    w = synth_weights(shape, "cuda", 77)
    rng = np.random.default_rng(9)
    toks = [1] + [int(t) for t in rng.integers(2, shape.vocab_size, n_prompt - 1)]
    exact = _decoder(shape, w)
    nxt_e = exact.prompt(toks)
    ke, ve = exact.kv_cache()
    le = exact.logits()
    fast = _decoder(shape, w)
    if split:
        fast.prompt(toks[:split])
    nxt_f = fast.prefill_w8(toks[split:], start_pos=split)
    kf, vf = fast.kv_cache()
    lf = fast.logits()
    n = len(toks)
    kv_worst = _rows_close((ke, ve), (kf, vf), n)
    d_logit = float(np.abs(le - lf).max())
    top2 = np.sort(le)[-2:]
    steps_worst = 0.0
    tok = nxt_e
    for pos in range(n, n + 16):
        a = exact.step(tok, pos)
        fast.step(tok, pos)
        steps_worst = max(steps_worst, float(np.abs(exact.logits() - fast.logits()).max()))
        tok = a
    print(f"[prefill_w8] {key} n={n} split={split} engine={engine}: max|dlogit| {d_logit:.3e}, "
          f"K/V max err/(rms+1e-3) {kv_worst:.3e}, 16 decode steps max|dlogit| {steps_worst:.3e}, "
          f"max|logit| {float(np.abs(le).max()):.3f}")
    assert d_logit <= TOL
    if top2[1] - top2[0] > 2 * TOL:
        assert nxt_e == nxt_f
    assert kv_worst <= TOL
    assert steps_worst <= TOL
    exact.close()
    fast.close()


def test_prefill_w8_golden(kllm_lib):
    """tests/golden/tiny_llama2_int8 (dim 64: one group per row): prefilling tokens[:t+1] gives the reference
    PyTorch logits of position t (dequantised weights) within 1e-4, for every t."""
    from kuiperllama_b200 import Decoder
    from kuiperllama_b200.checkpoint import read_checkpoint, to_device
    g = np.load(GOLDEN / "tiny_llama2_int8.npz")
    shape, w = read_checkpoint(str(GOLDEN / "tiny_llama2_int8.bin"), True)
    w = to_device(w)
    toks = [int(t) for t in g["tokens"]]
    worst = 0.0
    for t in range(len(toks)):
        dec = Decoder(shape, w)
        nxt = dec.prefill_w8(toks[:t + 1])
        lg = dec.logits()
        worst = max(worst, float(np.abs(lg - g["logits"][t]).max()))
        assert np.abs(lg - g["logits"][t]).max() < TOL, t
        top2 = np.sort(g["logits"][t])[-2:]
        if top2[1] - top2[0] > 2 * TOL:
            assert nxt == int(np.argmax(g["logits"][t]))
        dec.close()
    print(f"[prefill_w8] golden tiny_llama2_int8: max|dlogit| {worst:.3e}")


def test_prefill_w8_refuses_fp32(kllm_lib):
    from kuiperllama_b200 import SHAPES, Decoder, KllmError, synth_weights
    shape = SHAPES["small"]
    dec = Decoder(shape, synth_weights(shape, "cuda", 3))
    with pytest.raises(KllmError):
        dec.prefill_w8([1, 2, 3])
    dec.close()


@pytest.mark.parametrize("engine", ["persistent", "graph"])
def test_prefill_w8_is_deterministic(kllm_lib, monkeypatch, engine):
    from kuiperllama_b200 import SHAPES, synth_weights
    monkeypatch.setenv("KLLM_ENGINE", engine)
    shape = SHAPES["small-int8"]
    dec = _decoder(shape, synth_weights(shape, "cuda", 5))
    toks = [1] + list(range(7, 7 + 80))
    runs = []
    for _ in range(2):
        nxt = dec.prefill_w8(toks)
        k, v = dec.kv_cache()
        runs.append((nxt, dec.logits(), k, v))
    (n0, l0, k0, v0), (n1, l1, k1, v1) = runs
    assert n0 == n1
    for a, b in ((l0, l1), (k0, k1), (v0, v1)):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    dec.close()
