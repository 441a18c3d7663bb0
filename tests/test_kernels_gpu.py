"""-m gpu: every registry-level op of the C-ABI against
  (a) the reference's OWN CUDA kernels (oracle/_ref, compiled from a reference checkout for sm_100a):
      BIT-EXACT -- the design contract (DESIGN.md "Bit-exactness"); live when oracle/_ref is built,
      and always against their recorded outputs (tests/reference_outputs.py);
  (b) the CPU oracle: within fp32 reassociation tolerance (written at each assert).
Shapes follow the reference's tests (test_cu_*.cpp) plus the model shapes of BASELINE.json."""
import ctypes

import numpy as np
import pytest
import torch

from gpu_util import assert_bit_equal, dev, ptr, sync
from reference_outputs import check, live_reference

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ref():
    return live_reference("llama2")


@pytest.fixture(scope="module")
def ref_qwen():
    return live_reference("qwen2")


def rnd(shape, seed, scale=1.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.empty(shape, device="cuda", dtype=torch.float32).normal_(0, scale, generator=g)


# ---- matmul fp32 ----------------------------------------------------------------------------
def test_matmul_known_answers(kllm_lib, ref):
    # test_cu_matmul.cpp:78-105 ([1,1,-1] x 1..9 -> 0,3,6) and test_load.cpp:102-105
    x = dev(np.array([1, 1, -1], np.float32)); w = dev(np.arange(1, 10, dtype=np.float32).reshape(3, 3))
    out = torch.zeros(3, device="cuda")
    assert kllm_lib.kllm_gemv_f32(ptr(x), ptr(w), ptr(out), 3, 3, None) == 0
    sync()
    assert out.tolist() == [0, 3, 6]
    w = dev(np.arange(16 * 128, dtype=np.float32).reshape(16, 128)); x = torch.ones(128, device="cuda")
    out = torch.zeros(16, device="cuda")
    assert kllm_lib.kllm_gemv_f32(ptr(x), ptr(w), ptr(out), 128, 16, None) == 0
    sync()
    o = out.tolist()
    assert (o[0], o[1], o[14], o[15]) == (8128, 24512, 237504, 253888)


@pytest.mark.parametrize("M,K", [(4, 4), (288, 288), (288, 768), (768, 288), (896, 128), (896, 4864),
                                 (2048, 256), (2048, 2048), (2048, 5632), (5632, 2048),
                                 (4096, 4096), (11008, 4096), (4096, 11008), (2048, 32000),
                                 (130, 7), (3, 3)])
def test_matmul_bit_exact_vs_reference_cuda(kllm_lib, ref, oracle, M, K):
    x = rnd(M, 1 + M); w = rnd((K, M), 2 + K, 0.02)
    out = torch.zeros(K, device="cuda"); out_ref = torch.zeros(K, device="cuda")
    assert kllm_lib.kllm_gemv_f32(ptr(x), ptr(w), ptr(out), M, K, None) == 0
    if M % 4 == 0 or M < 4:  # the reference's float4 row loads need 16-byte aligned rows
        if ref:
            ref.L.kref_matmul_f32(ptr(x), ptr(w), ptr(out_ref), M, K, None)
        sync()
        check(out, out_ref if ref else None, f"matmul_f32/{K}x{M}", f"gemv_f32 {K}x{M} vs reference CUDA kernel")
    sync()
    if K * M <= 4096 * 4096:
        o_cuda_order = oracle.matmul(x.cpu().numpy(), w.cpu().numpy(), cuda_order=True)
        if M % 4 == 0 or M < 4:
            assert_bit_equal(out, o_cuda_order, "gemv_f32 vs oracle cuda-order model")
        strict = oracle.matmul(x.cpu().numpy(), w.cpu().numpy())
        # |x|~1, |w|~0.02, M terms: fp32 reassociation error << 1e-4 (north-star tolerance)
        assert np.abs(out.cpu().numpy() - strict).max() < 1e-4


# ---- matmul int8 ----------------------------------------------------------------------------
@pytest.mark.parametrize("M,K", [(128, 64), (256, 512), (4096, 4096), (11008, 4096), (4096, 11008),
                                 (4096, 32000), (320, 9)])
def test_matmul_w8_bit_exact(kllm_lib, ref, oracle, M, K):
    from kuiperllama_b200.decoder import quantize_q80
    w = rnd((K, M), 3 + K, 0.02); x = rnd(M, 4 + M)
    q, s = quantize_q80(w, 64)
    out = torch.zeros(K, device="cuda"); out_ref = torch.zeros(K, device="cuda")
    assert kllm_lib.kllm_gemv_w8(ptr(x), ptr(q), ptr(s), ptr(out), M, K, 64, None) == 0
    if ref:
        ref.L.kref_matmul_w8(ptr(x), ptr(q), ptr(s), ptr(out_ref), M, K, 64, None)
    sync()
    check(out, out_ref if ref else None, f"matmul_w8/{K}x{M}",
          f"gemv_w8 {K}x{M} vs reference CUDA kernel (int8 dequant arithmetic)")
    if K * M <= 4096 * 4096:
        oc = oracle.matmul_w8(x.cpu().numpy(), q.cpu().numpy(), s.cpu().numpy(), 64, cuda_order=True)
        assert_bit_equal(out, oc, "gemv_w8 vs oracle cuda-order model")
        st = oracle.matmul_w8(x.cpu().numpy(), q.cpu().numpy(), s.cpu().numpy(), 64)
        assert np.abs(out.cpu().numpy() - st).max() < 1e-4


# ---- rmsnorm ----------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [32, 480, 72480, 288, 896, 2048, 4096, 130])
def test_rmsnorm(kllm_lib, ref, ref_qwen, oracle, n):
    # sizes 480 / 32 / 72480 are the reference's own (test_cu_rmsnorm.cpp:7-119)
    x = rnd(n, 5 + n); w = rnd(n, 6 + n)
    for flavour, r in (("llama2", ref), ("qwen2", ref_qwen)):
        eps = oracle.eps(flavour)
        out = torch.zeros(n, device="cuda"); out_ref = torch.zeros(n, device="cuda")
        assert kllm_lib.kllm_rmsnorm_f32(ptr(x), ptr(w), ptr(out), n, eps, None) == 0
        if n % 4 == 0:
            if r:
                r.L.kref_rmsnorm(ptr(x), ptr(w), ptr(out_ref), n, None)
            sync()
            check(out, out_ref if r else None, f"rmsnorm/{flavour}/{n}", f"rmsnorm n={n} {flavour}")
        sync()
        cpu = oracle.rmsnorm(x.cpu().numpy(), w.cpu().numpy(), eps)
        assert np.abs(out.cpu().numpy() - cpu).max() < 1e-5 * max(1.0, np.abs(cpu).max())  # test_cu_rmsnorm.cpp tolerance
    # in place (llama3.cpp:726)
    xc = x.clone()
    assert kllm_lib.kllm_rmsnorm_f32(ptr(xc), ptr(w), ptr(xc), n, 1e-5, None) == 0
    out = torch.zeros(n, device="cuda")
    kllm_lib.kllm_rmsnorm_f32(ptr(x), ptr(w), ptr(out), n, 1e-5, None)
    sync()
    assert_bit_equal(xc, out, "rmsnorm in place")


# ---- add / swiglu -------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [4832, 62816, 5632, 7])
def test_add_and_swiglu(kllm_lib, ref, oracle, n):
    a = rnd(n, 7 + n, 3.0); b = rnd(n, 8 + n)
    out = torch.zeros(n, device="cuda"); out_ref = torch.zeros(n, device="cuda")
    assert kllm_lib.kllm_add_f32(ptr(a), ptr(b), ptr(out), n, None) == 0
    if ref:
        ref.L.kref_add(ptr(a), ptr(b), ptr(out_ref), n, None)
    sync()
    check(out, out_ref if ref else None, f"add/{n}", "add")
    assert kllm_lib.kllm_swiglu_f32(ptr(a), ptr(b), ptr(out), n, None) == 0
    if ref:
        ref.L.kref_swiglu(ptr(a), ptr(b), ptr(out_ref), n, None)
    sync()
    check(out, out_ref if ref else None, f"swiglu/{n}", "swiglu")
    cpu = oracle.swiglu(a.cpu().numpy(), b.cpu().numpy())
    assert np.abs(out.cpu().numpy() - cpu).max() < 1e-5  # test_cu_swiglu.cpp tolerance


# ---- sin/cos table + rope -----------------------------------------------------------------------
@pytest.mark.parametrize("flavour,head_size,seq_len", [("llama2", 64, 2048), ("llama2", 48, 256),
                                                       ("llama2", 128, 512), ("qwen2", 64, 4096)])
def test_sincos_table(kllm_lib, ref, ref_qwen, oracle, flavour, head_size, seq_len):
    from kuiperllama_b200 import FLAVOURS
    r = ref if flavour == "llama2" else ref_qwen
    s = torch.zeros(seq_len * head_size, device="cuda"); c = torch.zeros_like(s)
    sr = torch.zeros_like(s); cr = torch.zeros_like(s)
    assert kllm_lib.kllm_sincos_init(head_size, seq_len, FLAVOURS[flavour], ptr(s), ptr(c), None) == 0
    if r:
        r.L.kref_sincos(head_size, seq_len, ptr(sr), ptr(cr), None)
    sync()
    key = f"sincos/{flavour}/{head_size}x{seq_len}"
    check(s, sr if r else None, key + "/sin", "sin table")
    check(c, cr if r else None, key + "/cos", "cos table")
    so, co = oracle.sincos(head_size, seq_len, flavour)
    # device powf/sinf/cosf vs libm at arguments up to seq_len: absolute 2e-4 (values in [-1,1])
    assert np.abs(s.cpu().numpy() - so.ravel()).max() < 2e-4
    assert np.abs(c.cpu().numpy() - co.ravel()).max() < 2e-4


@pytest.mark.parametrize("flavour,dim,kv_dim,head_size", [("llama2", 2048, 256, 64), ("llama2", 288, 288, 48),
                                                          ("llama2", 4096, 4096, 128), ("qwen2", 896, 128, 64),
                                                          ("qwen2", 2048, 2048, 64)])
def test_rope(kllm_lib, ref, ref_qwen, oracle, flavour, dim, kv_dim, head_size):
    from kuiperllama_b200 import FLAVOURS
    r = ref if flavour == "llama2" else ref_qwen
    seq_len = 64
    s = torch.zeros(seq_len * head_size, device="cuda"); c = torch.zeros_like(s)
    kllm_lib.kllm_sincos_init(head_size, seq_len, FLAVOURS[flavour], ptr(s), ptr(c), None)
    for pos in (0, 1, 37, 63):
        q0 = rnd(dim, 9 + pos); k0 = rnd(kv_dim, 10 + pos)
        q, k = q0.clone(), k0.clone()
        assert kllm_lib.kllm_rope_f32(FLAVOURS[flavour], dim, kv_dim, head_size, ptr(q), ptr(k), pos,
                                      ptr(s), ptr(c), None) == 0
        # the reference's half-split kernel writes one pair past the end of q (rope_kernel.cu:13,59):
        # give it a padded buffer so the overrun stays inside our allocation.
        qr = torch.zeros(dim + head_size, device="cuda"); qr[:dim] = q0
        kr = k0.clone()
        if r:
            r.L.kref_rope(dim, kv_dim, head_size, ptr(qr), ptr(kr), pos, ptr(s), ptr(c), seq_len, None)
        sync()
        key = f"rope/{flavour}/{dim}x{kv_dim}x{head_size}/pos{pos}"
        check(q, qr[:dim] if r else None, key + "/q", f"rope q {flavour} pos={pos}")
        check(k, kr if r else None, key + "/k", f"rope k {flavour} pos={pos}")
        qo, ko = oracle.rope(flavour, q0.cpu().numpy(), k0.cpu().numpy(), pos,
                             s.cpu().numpy(), c.cpu().numpy(), head_size)
        assert np.abs(q.cpu().numpy() - qo).max() < 1e-5 and np.abs(k.cpu().numpy() - ko).max() < 1e-5


# ---- attention ------------------------------------------------------------------------------------
@pytest.mark.parametrize("heads,kv_heads,head_size,seq_len,positions", [
    (6, 6, 48, 256, [0, 1, 5, 255]), (32, 4, 64, 2048, [0, 31, 32, 33, 300, 1023, 2047]),
    (14, 2, 64, 512, [0, 257, 511]), (32, 32, 128, 1024, [0, 100, 1023]),
    (14, 2, 64, 4096, [0, 1023, 4095])])  # Qwen2.5-0.5B geometry (kv_mul 7) to pos 1023 and beyond
def test_mha_decode(kllm_lib, ref, oracle, heads, kv_heads, head_size, seq_len, positions):
    kv_dim = kv_heads * head_size; kv_mul = heads // kv_heads; L = 2; layer = 1
    kc = rnd((L, seq_len, kv_dim), 11); vc = rnd((L, seq_len, kv_dim), 12)
    for pos in positions:
        q = rnd(heads * head_size, 13 + pos)
        out = torch.zeros(heads * head_size, device="cuda"); out_ref = torch.zeros_like(out)
        sc = torch.zeros(heads * seq_len, device="cuda"); sc_ref = torch.zeros_like(sc)
        assert kllm_lib.kllm_mha_decode_f32(pos, heads, layer, seq_len, kv_dim, kv_mul, head_size, ptr(out),
                                            ptr(q), ptr(sc), ptr(kc), ptr(vc), None) == 0
        if ref:
            ref.L.kref_mha(pos, heads, layer, seq_len, kv_dim, kv_mul, head_size, ptr(out_ref), ptr(q),
                           ptr(sc_ref), ptr(kc), ptr(vc), L, None)
        sync()
        key = f"mha/{heads}x{kv_heads}x{head_size}x{seq_len}/pos{pos}"
        check(out, out_ref if ref else None, key + "/out", f"mha out pos={pos}")
        check(sc.view(heads, seq_len)[:, :pos + 1], sc_ref.view(heads, seq_len)[:, :pos + 1] if ref else None,
              key + "/probabilities", f"softmax probabilities pos={pos}")
        if pos <= 300:
            oc, _ = oracle.mha(pos, heads, layer, seq_len, kv_dim, kv_mul, head_size, q.cpu().numpy(),
                               kc.cpu().numpy(), vc.cpu().numpy())
            assert np.abs(out.cpu().numpy() - oc).max() < 1e-5


# ---- embedding / argmax -----------------------------------------------------------------------------
def test_embedding(kllm_lib, ref, oracle):
    # test_cu_emb.cpp:6-31: arange table, token 1, dim 512
    table = dev(np.arange(4 * 512, dtype=np.float32).reshape(4, 512))
    toks = dev(np.array([1], np.int32)); out = torch.zeros(512, device="cuda")
    assert kllm_lib.kllm_embedding_f32(ptr(toks), 1, ptr(table), ptr(out), 512, 4, None) == 0
    sync()
    assert np.array_equal(out.cpu().numpy(), 512 + np.arange(512, dtype=np.float32))
    table = rnd((1000, 288), 14); ids = np.array([0, 999, 5, 5, 1000, -1, 17], np.int32)
    out = torch.full((7, 288), -7.0, device="cuda"); out_ref = torch.full((7, 288), -7.0, device="cuda")
    assert kllm_lib.kllm_embedding_f32(ptr(dev(ids)), 7, ptr(table), ptr(out), 288, 1000, None) == 0
    good = ids.copy(); good[good < 0] = 1000  # the reference kernel only guards token >= vocab
    arr = (ctypes.c_int32 * 7)(*good.tolist())
    if ref:
        ref.L.kref_embedding(arr, 7, ptr(table), ptr(out_ref), 288, 1000, None)
    sync()
    check(out, out_ref if ref else None, "embedding/1000x288", "embedding rows (out-of-range ids leave the row untouched)")


def test_argmax(kllm_lib, ref, oracle):
    for n, seed in [(32000, 1), (151936, 2), (5, 3), (1024, 4), (1025, 5)]:
        x = rnd(n, seed)
        got = kllm_lib.kllm_argmax_f32_sync(ptr(x), n, None)
        assert got == int(torch.argmax(x)) == oracle.argmax(x.cpu().numpy())
        check([got], [ref.L.kref_argmax(ptr(x), n, None)] if ref else None, f"argmax/{n}", f"argmax n={n}")
    x = torch.zeros(32000, device="cuda"); x[[77, 5000, 31999]] = 3.0  # ties -> lowest index
    got = kllm_lib.kllm_argmax_f32_sync(ptr(x), 32000, None)
    assert got == 77
    check([got], [ref.L.kref_argmax(ptr(x), 32000, None)] if ref else None, "argmax/ties", "argmax ties")
    x = torch.full((4096,), -5.0, device="cuda")  # all negative, all equal
    assert kllm_lib.kllm_argmax_f32_sync(ptr(x), 4096, None) == 0


# ---- fused GEMV entry point ---------------------------------------------------------------------------
def test_gemv_fused_matches_op_chain(kllm_lib, ref_qwen, oracle):
    """norm -> q|k|v(+bias), w1|w3 -> swiglu, wo + residual: the fused launch must equal the chain
    of reference kernels it replaces, bit for bit."""
    from kuiperllama_b200 import GemvJob
    dim, kvd, hid = 896, 128, 4864
    x = rnd(dim, 20); nw = rnd(dim, 21) + 1.0
    wq, wk, wv = rnd((dim, dim), 22, 0.02), rnd((kvd, dim), 23, 0.02), rnd((kvd, dim), 24, 0.02)
    bq, bk, bv = rnd(dim, 25, 0.02), rnd(kvd, 26, 0.02), rnd(kvd, 27, 0.02)
    q, k, v = (torch.zeros(n, device="cuda") for n in (dim, kvd, kvd))
    nout = torch.zeros(dim, device="cuda")
    job = GemvJob()
    job.x = x.data_ptr(); job.norm_w = nw.data_ptr(); job.norm_eps = 1e-6; job.norm_out = nout.data_ptr()
    job.in_dim = dim; job.n_seg = 3
    for i, (w, b, o, rows) in enumerate([(wq, bq, q, dim), (wk, bk, k, kvd), (wv, bv, v, kvd)]):
        job.seg[i].w = w.data_ptr(); job.seg[i].bias = b.data_ptr(); job.seg[i].out = o.data_ptr(); job.seg[i].rows = rows
    assert kllm_lib.kllm_gemv_fused(ctypes.byref(job), None) == 0
    rq = ref_qwen
    xn = torch.zeros(dim, device="cuda")
    if rq:
        rq.L.kref_rmsnorm(ptr(x), ptr(nw), ptr(xn), dim, None)
    for w, b, o, rows, name in [(wq, bq, q, dim, "q"), (wk, bk, k, kvd, "k"), (wv, bv, v, kvd, "v")]:
        t = torch.zeros(rows, device="cuda")
        if rq:
            rq.L.kref_matmul_f32(ptr(xn), ptr(w), ptr(t), dim, rows, None)
            rq.L.kref_add(ptr(t), ptr(b), ptr(t), rows, None)  # matmul.cpp:74-77
        sync()
        check(o, t if rq else None, f"gemv_fused/{name}", f"fused qkv: {name}")
    check(nout, xn if rq else None, "gemv_fused/norm_out", "fused norm_out")
    # w1|w3 -> swiglu
    w1, w3 = rnd((hid, dim), 28, 0.02), rnd((hid, dim), 29, 0.02)
    h = torch.zeros(hid, device="cuda")
    job = GemvJob(); job.x = x.data_ptr(); job.norm_w = nw.data_ptr(); job.norm_eps = 1e-6
    job.in_dim = dim; job.n_seg = 2; job.swiglu_pair = 1
    job.seg[0].w = w1.data_ptr(); job.seg[0].out = h.data_ptr(); job.seg[0].rows = hid
    job.seg[1].w = w3.data_ptr(); job.seg[1].rows = hid
    assert kllm_lib.kllm_gemv_fused(ctypes.byref(job), None) == 0
    a = torch.zeros(hid, device="cuda"); b = torch.zeros(hid, device="cuda")
    if rq:
        rq.L.kref_matmul_f32(ptr(xn), ptr(w1), ptr(a), dim, hid, None)
        rq.L.kref_matmul_f32(ptr(xn), ptr(w3), ptr(b), dim, hid, None)
        rq.L.kref_swiglu(ptr(a), ptr(b), ptr(a), hid, None)
    sync()
    check(h, a if rq else None, "gemv_fused/w1w3_swiglu", "fused w1|w3 swiglu")
    # w2 + residual (in place on the residual stream)
    w2 = rnd((dim, hid), 30, 0.02); res = rnd(dim, 31); res_ref = res.clone()
    job = GemvJob(); job.x = h.data_ptr(); job.in_dim = hid; job.n_seg = 1
    job.seg[0].w = w2.data_ptr(); job.seg[0].out = res.data_ptr(); job.seg[0].rows = dim
    job.residual = res.data_ptr()
    assert kllm_lib.kllm_gemv_fused(ctypes.byref(job), None) == 0
    t = torch.zeros(dim, device="cuda")
    if rq:
        rq.L.kref_matmul_f32(ptr(a), ptr(w2), ptr(t), hid, dim, None)
        rq.L.kref_add(ptr(res_ref), ptr(t), ptr(res_ref), dim, None)  # llama3.cpp:719
    sync()
    check(res, res_ref if rq else None, "gemv_fused/w2_residual", "fused w2 + residual")


def test_streams_and_launch_counter(kllm_lib):
    s = torch.cuda.Stream()
    before = kllm_lib.kllm_launch_count()
    a = rnd(4832, 40); b = rnd(4832, 41); out = torch.zeros(4832, device="cuda")
    with torch.cuda.stream(s):
        assert kllm_lib.kllm_add_f32(ptr(a), ptr(b), ptr(out), 4832, ctypes.c_void_p(s.cuda_stream)) == 0
    s.synchronize()
    assert torch.equal(out, a + b)  # test_cu_add.cpp "stream" variants
    assert kllm_lib.kllm_launch_count() == before + 1
