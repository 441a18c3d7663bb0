#!/usr/bin/env python
"""Prompt throughput of Llama-2-7B int8: position-by-position prompt() against batched prefill_w8()
(kllm_decoder_prefill_w8, tcgen05 kind::i8 GEMMs), and kllm_gemm_w8 alone at the model's projection shapes.
Needs a CUDA device; prints one JSON line (and writes it to --out when given).

    python tools/prefill_bench.py --out /tmp/prefill_w8_bench.json

Prompt rates: host clock around each call, which ends in a device synchronise; warm-up first, median and
spread (min, max) of --reps repetitions.  The same decoder and seeded weights serve both paths, and the
max |dlogit| between them is taken from the timed runs.  GEMM times: CUDA events over --gemm-iters launches,
cycling through enough weight copies to overflow the 126 MB L2, so weights come from HBM.  Floors: int8 ops
over the data sheet's dense int8 rate for one GPU, weight bytes over the data sheet's HBM bandwidth (both
are ceilings the card does not reach); `floor_share` = the larger floor / measured time.
"""
import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

DENSE_INT8_OPS = 4.5e15  # HGX B200 data sheet, dense int8, per GPU
HBM_BYTES_PER_S = 7.7e12
GEMM_SHAPES = [(4096, 4096), (4096, 11008), (11008, 4096), (4096, 32000)]  # K x N


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in out.split(","))
    return {"name": name, "power_limit": power}


def timed(fn, reps):
    fn()  # warm-up
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        times.append(time.perf_counter() - t0)
    return times


def bench_gemm(lib, T, K, N, iters):
    import ctypes
    import torch
    g = torch.Generator(device="cuda").manual_seed(K + N)
    copies = max(1, -(-300_000_000 // (N * K)))  # > 2 x L2 of weights in rotation
    ws_ = [torch.randint(-127, 128, (N, K), device="cuda", generator=g, dtype=torch.int8) for _ in range(copies)]
    sc = torch.rand(N, K // 64, device="cuda", generator=g) * 1e-4
    x = torch.randn(T, K, device="cuda", generator=g)
    out = torch.empty(T, N, device="cuda")
    work = torch.empty(3 * T * K + 4 * (K // 64) * ((T + 63) // 64 * 64), dtype=torch.uint8, device="cuda")
    p = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731

    def run(i):
        rc = lib.kllm_gemm_w8(p(x), p(ws_[i % copies]), p(sc), p(out), p(work), T, K, N, None)
        assert rc == 0, rc

    for i in range(copies + 2):
        run(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        run(i)
    e1.record()
    torch.cuda.synchronize()
    sec = e0.elapsed_time(e1) / 1e3 / iters
    ops = 3 * 2 * T * N * K
    wbytes = N * K + N * (K // 64) * 4
    t_ops, t_bytes = ops / DENSE_INT8_OPS, wbytes / HBM_BYTES_PER_S
    return {"T": T, "K": K, "N": N, "us": round(sec * 1e6, 2), "int8_tensor_ops": ops,
            "int8_tops": round(ops / sec / 1e12, 1), "weight_bytes": wbytes,
            "weight_gb_per_s": round(wbytes / sec / 1e9, 1),
            "floor_binding": "int8 ops" if t_ops >= t_bytes else "HBM bytes",
            "floor_share": round(max(t_ops, t_bytes) / sec, 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="llama2-7b-int8")
    ap.add_argument("--lengths", default="128,512,2000")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--gemm-iters", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        sys.exit("prefill_bench.py needs a CUDA device")
    from kuiperllama_b200 import SHAPES, Decoder, load_library, synth_weights
    lib = load_library()
    result = {"card": card(), "workload": a.workload}

    shape = SHAPES[a.workload]
    w = synth_weights(shape, "cuda", 1234)
    dec = Decoder(shape, w)
    result["engine"] = dec.engine
    rng = np.random.default_rng(7)
    prompts = []
    for n in (int(s) for s in a.lengths.split(",")):
        toks = [1] + [int(t) for t in rng.integers(2, shape.vocab_size, n - 1)]
        t_prompt = timed(lambda: dec.prompt(toks), a.reps)
        l_prompt = dec.logits()
        t_w8 = timed(lambda: dec.prefill_w8(toks), a.reps)
        l_w8 = dec.logits()
        mp, mw = statistics.median(t_prompt), statistics.median(t_w8)
        prompts.append({
            "tokens": n,
            "prompt_tok_s": round(n / mp, 1), "prompt_s": {"median": round(mp, 5), "min": round(min(t_prompt), 5),
                                                             "max": round(max(t_prompt), 5)},
            "prefill_w8_tok_s": round(n / mw, 1), "prefill_w8_s": {"median": round(mw, 5),
                                                                   "min": round(min(t_w8), 5),
                                                                   "max": round(max(t_w8), 5)},
            "speedup": round(mp / mw, 2),
            "max_abs_dlogit": float(np.abs(l_prompt - l_w8).max()),
            "max_abs_logit": float(np.abs(l_prompt).max()),
        })
    result["prompt"] = prompts
    dec.close()
    del w
    torch.cuda.empty_cache()

    gemms = [bench_gemm(lib, 256, K, N, a.gemm_iters) for K, N in GEMM_SHAPES]
    result["gemm_w8_T256"] = gemms
    # GEMM time of one 256-token block through all layers: wq wk wv wo (4096 x 4096), w1 w3 (4096 x 11008),
    # w2 (11008 x 4096); the classifier runs once per prompt through the GEMV
    us = {(g["K"], g["N"]): g["us"] for g in gemms}
    block_us = shape.layer_num * (4 * us[(4096, 4096)] + 2 * us[(4096, 11008)] + us[(11008, 4096)])
    result["gemm_us_per_256_block"] = round(block_us, 1)
    for p in prompts:  # share of prefill_w8's time the projections take, scaled by tokens / 256
        p["gemm_share_est"] = round(block_us * p["tokens"] / 256 / 1e6 / p["prefill_w8_s"]["median"], 3)
    line = json.dumps(result)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
