#!/usr/bin/env python
"""bench.py -- decode tokens/s of the B200-native KuiperLLama hot path (BASELINE.json `metric`).

One "step" = one greedy decode position (one token, batch 1) of the workload's model through the
device-resident decoder (libkllm_b200.so).  The metric is quoted on context 1 -> 1024, so the
context is NOT tied to --steps:

  1. an untimed pre-pass decodes positions 0..1023 (fills the KV cache, doubles as warm-up and as the
     parity record: every later window must reproduce its token ids);
  2. the timed region is EXACTLY --steps positions.  --steps >= 1024: positions 0..steps-1 in one
     run (the true 1->1024 mean).  Fewer steps: the positions are spread over the context as up to
     16 equal windows placed evenly between position 0 and 1023 (cost is linear in the position, so
     evenly spaced samples give the 1->1024 mean);  config.windows lists them;
  3. the whole timed region is repeated --reps times and the MEDIAN repetition is reported
     (per window: CUDA events on the decoder's stream, max over ranks);
  4. `by_position` adds tokens/s in short windows at positions 1, 256 and 1023.

--dump-outputs DIR writes what the timed path returned at its last timed step (last window of the last
repetition) as DIR/logits.npy (float32 [vocab]) and DIR/next_token.npy (float64 [1], the greedy id).
Weights and token inputs are seeded, so runs with the same arguments see identical inputs and two builds
can be compared output for output.

  value   device-resident loop: tokens fed back on the GPU, no host round trip inside a window.
  e2e     the same positions through the reference-facing call kllm_decoder_step() with HOST
          buffers: per step the token id + position go host->device (pinned, 16 B), the greedy id
          comes back (16 B) and the host synchronises -- LLama2Model::predict + post_processing
          (llama3.cpp:642-650,733-745).
  roofline      the persistent megakernel (the only kernel of the step): algorithmic weight bytes
                per launch / event-timed launch duration vs MEASURED_PEAKS.json.
  cpu_baseline  the CPU restatement of the reference path (oracle/) on the box's host cores.

Workloads.  1 GPU on a single-GPU box: BASELINE.json configs[1], TinyLlama-1.1B fp32.  Under
tensor parallelism (--gpus N > 1) and for the N = 1 point of the same series (any run on a box
with several GPUs): the model the metric names for 1/2/4/8 GPUs, Llama-2-7B int8 (configs[2]);
the fp32 Llama-2-7B of configs[4] is measured in the same run and reported under `secondary`.
--workload overrides.

--impl reference       the reference's CPU implementation of the path (oracle port; the reference's
                       CMake build needs Armadillo/glog/gtest/sentencepiece, none installed).
--impl reference-cuda  the reference's own CUDA kernels + model code (oracle/_ref, compiled from the
                       checkout KUIPER_REFERENCE_DIR names, for sm_100a) timed on the same GPU: the
                       "reference GPU" row.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "decode_tokens_per_s"
CONTEXT = 1024  # the metric's context: 1 -> 1024
# BASELINE.md section 1: the one number the reference publishes for this metric -- TinyLlama-1.1B fp32,
# batch 1, its CUDA backend on an RTX 3060 Laptop GPU (readme.md:25).  Other workloads: none.
PUBLISHED_TOK_S = {"tinyllama-1.1b": 60.34}
WORKLOAD_NAMES = {
    "tinyllama-1.1b": "TinyLlama-1.1B fp32 greedy decode, batch 1 (BASELINE.json configs[1])",
    "llama2-7b-int8": "Llama-2-7B int8 g64 (export.py --version 3) greedy decode, batch 1 (configs[2]; metric's 1/2/4/8-GPU model)",
    "qwen2.5-0.5b": "Qwen2.5-0.5B fp32 greedy decode, batch 1 (configs[3])",
    "llama2-7b": "Llama-2-7B fp32 greedy decode, batch 1 (configs[4])",
    "stories15m": "stories15M fp32 greedy decode, batch 1 (configs[0])",
    "small": "synthetic dim-288 3-layer model (debug)",
}


def vs_baseline(workload, tok_s):
    ref = PUBLISHED_TOK_S.get(workload)
    return tok_s / ref if ref else None


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1024)
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-cuda"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOAD_NAMES),
                    help="default: tinyllama-1.1b on a single-GPU box at --gpus 1, else llama2-7b-int8")
    ap.add_argument("--reps", type=int, default=5, help="repetitions of the timed region; the median is reported")
    ap.add_argument("--numerics", default="fast", choices=["fast", "exact"],
                    help="fast (default): toleranced mode, |dlogit| <= 1e-4 vs the reference (tests/test_decoder_gpu.py); "
                         "exact: every reduction in the reference's order, bit-identical logits.  The fast line "
                         "carries the exact mode's numbers under \"exact\"")
    ap.add_argument("--no-exact", action="store_true", help="skip the exact-mode leg of a --numerics fast run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="N>1: skip the fp32 Llama-2-7B line (configs[4])")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--seed", type=int, default=None)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the timed path's outputs of its last step to DIR/*.npy (--impl ours)")
    return ap.parse_args()


SEEDS = {"stories15m": 1234, "tinyllama-1.1b": 1235, "llama2-7b-int8": 1236, "qwen2.5-0.5b": 1237,
         "llama2-7b": 1238, "small": 1239}


def default_workload(n_gpus):
    """configs[1] on one GPU of a single-GPU box; the metric's 1/2/4/8-GPU model otherwise."""
    if n_gpus > 1:
        return "llama2-7b-int8"
    try:
        import torch
        if torch.cuda.is_available() and torch.cuda.device_count() > 1:
            return "llama2-7b-int8"
    except Exception:
        pass
    return "tinyllama-1.1b"


def plan_windows(steps, ctx):
    """[(start_pos, n)] with sum(n) == steps, spread evenly over the context 1 -> ctx."""
    if steps >= ctx:
        return [(0, steps)]
    nw = max(1, min(16, steps // 4))
    base, extra = divmod(steps, nw)
    sizes = [base + (1 if i < extra else 0) for i in range(nw)]
    if nw == 1:
        return [((ctx - sizes[0]) // 2, sizes[0])]
    return [(round(i * (ctx - sizes[i]) / (nw - 1)), sizes[i]) for i in range(nw)]


# ------------------------------------------------------------------------------------------
# clocks: sample nvidia-smi DURING the timed region (started BEFORE the barrier that opens it)
# ------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for t, r in self.rows if t0 <= t <= t1 + 0.2] or [r for _, r in self.rows]
        for r in rows:
            parts = [p.strip() for p in r.split(",")]
            try:
                sm.append(float(parts[0])); smax = max(smax, float(parts[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return None
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------
def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            d = json.loads(p.read_text())
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, torch copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(workload, kernel_key):
    """DRAM traffic (dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture)
    of a kernel, from the committed summary profiles/dominant_kernel_traffic.json, or None."""
    p = ROOT / "profiles" / "dominant_kernel_traffic.json"
    if p.exists():
        try:
            return json.loads(p.read_text()).get(workload, {}).get(kernel_key)
        except Exception:
            return None
    return None


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


# ------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's CPU path
# ------------------------------------------------------------------------------------------
def cpu_reference_run(shape, w, max_steps, budget_s, first_token=1):
    """Time the CPU restatement of the reference path on this box's host cores: up to `max_steps`
    consecutive decode positions from context 1, stopping early at `budget_s` seconds.

    Threads are set through the BLAS's / OpenMP's own API (an inherited OMP_NUM_THREADS=1, which
    torchrun exports, must not serialise the arm).  A multi-threaded sgemv can be SLOWER than a
    single thread on a box whose cores are shared or throttled, so the matmul back-end (OpenBLAS
    sgemv as the reference's Armadillo would call, or OpenMP row-parallel loops) and the thread
    count are picked by a short calibration on the model's own first step, and reported."""
    from kuiperllama_b200.checkpoint import write_checkpoint
    from oracle.binding import Oracle, find_openblas
    ckpt_dir = "/dev/shm" if os.path.isdir("/dev/shm") else "/tmp"
    path = os.path.join(ckpt_dir, f"kllm_bench_{os.getpid()}.bin")
    o = Oracle()
    blas = find_openblas()
    ncores = host_cores()
    try:
        write_checkpoint(path, shape, w)
        m = o.open_model(path, shape.group_size > 0, shape.flavour)
        m.step(first_token, 0, want_logits=False)  # page in the mmap
        cands = []
        # most threads first: a 7B int8 step takes ~17 s on ONE core, and the calibration must not spend
        # its budget there (it stops after 40 s, keeping the best setting seen)
        threads = sorted({1, max(1, ncores // 4), max(1, ncores // 2), ncores}, reverse=True)
        t_cal = time.perf_counter()
        backends = ([("openblas", blas)] if blas and shape.group_size == 0 else []) + [("openmp", None)]
        best = None
        for name, lib in backends:
            if not o.use_fast_matmul(True, lib) and lib:
                continue
            for n in threads:
                got = o.set_num_threads(n)
                t0 = time.perf_counter()
                m.step(first_token, 0, want_logits=False)
                dt = time.perf_counter() - t0
                cands.append((name, n, got, dt))
                if best is None or dt < best[3]:
                    best = (name, n, got, dt, lib)
                if time.perf_counter() - t_cal > 40.0:
                    break
            if time.perf_counter() - t_cal > 40.0:
                break
        name, n, got, _, lib = best
        o.use_fast_matmul(True, lib)
        o.set_num_threads(n)
        tok, pos, done, t0 = first_token, 0, 0, time.perf_counter()
        while done < max_steps and pos < shape.seq_len:
            tok, _ = m.step(tok, pos, want_logits=False)
            pos += 1; done += 1
            dt = time.perf_counter() - t0
            if dt >= budget_s:
                break
        m.close()
        o.use_fast_matmul(False)
    finally:
        if os.path.exists(path):
            os.remove(path)
    back = f"OpenBLAS sgemv ({os.path.basename(lib)}, {got} BLAS threads)" if name == "openblas" else \
        f"OpenMP row-parallel loops ({n} threads)"
    return {"value": done / dt, "unit": "tokens/s", "cores": n, "host_cores": ncores, "kind": "port",
            "steps": done,
            "sample": f"{done} consecutive decode positions (context 1..{pos}) of {shape.name}, {back}, {dt:.1f} s; "
                      f"back-end and thread count picked by calibration on one step "
                      f"({', '.join(f'{a}x{b}:{d * 1e3:.0f}ms' for a, b, _, d in cands)}); "
                      "oracle/kuiper_oracle.c restating kuiper/source/op/kernels/cpu/*.cpp + llama3.cpp"}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path (restated port), rank 0 only."""
    if rank != 0:
        return
    import torch
    from kuiperllama_b200 import SHAPES, synth_weights
    shape = SHAPES[args.workload]
    w = synth_weights(shape, "cuda" if torch.cuda.is_available() else "cpu", args.seed)
    res = cpu_reference_run(shape, w, args.steps, budget_s=150.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": "tokens/s",
        "n_gpus": args.gpus, "steps": res["steps"], "warmup": args.warmup,
        "ms_per_step": 1e3 / res["value"], "higher_is_better": True, "scaling": "strong",
        "vs_baseline": vs_baseline(args.workload, res["value"]),
        "dtype": "f32" if shape.group_size == 0 else "int8w/f32",
        "data": "synthetic random-init weights (tools/model.py init, seed %d), greedy decode from token 1" % args.seed,
        "config": {"workload": WORKLOAD_NAMES[args.workload], "shape": shape.name, "batch": 1,
                   "context": f"1->{res['steps']} (consecutive positions from context 1; the CPU path's cost "
                              "per position is dominated by the weights, not the context)",
                   "requested_steps": args.steps, "parallelism": "host CPU"},
        "cpu_baseline": res,
        "e2e": {"value": res["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def run_reference_cuda(args, rank, world):
    """--impl reference-cuda: oracle/_ref -- the reference's own .cu/.cpp compiled for sm_100a --
    decoding the same synthetic checkpoint on this GPU through LLama2Model::predict (rank 0)."""
    if rank != 0:
        return
    import numpy as np
    import torch
    from kuiperllama_b200 import SHAPES, synth_weights
    from kuiperllama_b200.checkpoint import write_checkpoint
    from oracle.binding import REF_SO, RefCuda
    shape = SHAPES[args.workload]
    base = {"impl": "reference-cuda", "metric": METRIC, "unit": "tokens/s", "n_gpus": 1}
    if not REF_SO.exists() or shape.flavour != "llama2":
        emit({**base, "unavailable": "oracle/_ref has no model build for this workload "
                          "(QWEN2 flavour needs absl/re2 for its tokenizer)" if REF_SO.exists() else "oracle/_ref not built"})
        return
    w = synth_weights(shape, "cuda", args.seed)
    path = os.path.join("/dev/shm" if os.path.isdir("/dev/shm") else "/tmp", f"kllm_refcuda_{os.getpid()}.bin")
    try:
        write_checkpoint(path, shape, w)
        del w
        torch.cuda.empty_cache()
        ref = RefCuda("llama2")
        h = ref.L.kref_model_create(path.encode(), int(shape.group_size > 0))
        assert h, "reference LLama2Model::init failed"
        K = min(args.steps, CONTEXT)
        tok = 1
        for pos in range(min(args.warmup, 8)):
            tok = ref.L.kref_model_step(h, tok, pos, None, shape.vocab_size)
        torch.cuda.synchronize()
        tok, t0 = 1, time.perf_counter()
        for pos in range(K):  # demo/main.cpp:18-41: one predict() per position, host-synchronous
            tok = ref.L.kref_model_step(h, tok, pos, None, shape.vocab_size)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        ref.L.kref_model_destroy(h)
    finally:
        if os.path.exists(path):
            os.remove(path)
    emit({**base, "value": K / dt, "steps": K, "ms_per_step": dt / K * 1e3, "higher_is_better": True,
                      "dtype": "f32" if shape.group_size == 0 else "int8w/f32",
                      "config": {"workload": WORKLOAD_NAMES[args.workload], "shape": shape.name, "context": f"1->{K}",
                                 "batch": 1, "what": "the reference's own CUDA backend (kuiper/source/op/kernels/cuda/*.cu "
                                 "+ model/llama3.cpp, unmodified, nvcc 12.9 sm_100a) on this GPU, wall clock of the predict loop"},
                      "roofline_frac_of_measured_hbm": shape.weight_bytes_per_token() * K / dt / 1e9 / measured_peaks()[0]})


_REAL_STDOUT = None


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def _leave_process_group():
    try:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
class Bench:
    """One workload on `world` GPUs: build, pre-pass, timed windows, e2e, per-position numbers."""

    def __init__(self, args, rank, world, workload, stream, lib, numerics=None):
        import torch
        from kuiperllama_b200 import SHAPES, Decoder, synth_weights
        self.torch, self.args, self.rank, self.world, self.workload, self.lib = torch, args, rank, world, workload, lib
        self.shape = shape = SHAPES[workload]
        self.stream = stream
        seed = args.seed if (args.seed is not None and workload == args.workload) else SEEDS.get(workload, 1234)
        self.seed = seed
        self.comm = None
        self.local = shape
        self.parity = None
        self.numerics = numerics = numerics or args.numerics
        if world > 1:
            import torch.distributed as dist
            from kuiperllama_b200.tensor_parallel import Comm, comm_words, local_shape, make_tp_decoder
            self.comm = Comm(comm_words(shape, world))  # room for vocab / world words: classifier sharded by vocabulary
            full = synth_weights(shape, "cuda", seed)  # same seed on every rank -> same model
            self.dec = make_tp_decoder(shape, full, self.comm, stream.cuda_stream, numerics=numerics)
            self.w, self.local = self.dec.weights, local_shape(shape, world, rank)
            self.parity = self._tp_parity(full, dist)
            del full
            torch.cuda.empty_cache()
        else:
            self.w = synth_weights(shape, "cuda", seed)
            self.dec = Decoder(shape, self.w, stream=stream.cuda_stream, numerics=numerics)
        self.engine = self.dec.engine
        self.launches_per_step = self.dec.launches_per_step

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        self.torch.cuda.synchronize()

    def _tp_parity(self, full, dist, steps=8, tol=1e-4):
        """SCALE's own parity bit: the tensor-parallel decoder, teacher-forced with the UNSHARDED
        decoder's tokens, must give logits within the north-star tolerance (1e-4) of the unsharded
        single-GPU decoder at every position and the same greedy id wherever the top-2 margin
        exceeds 2e-4 (the split only changes the summation tree of the two row-parallel matmuls)."""
        import numpy as np
        from kuiperllama_b200 import Decoder
        torch = self.torch
        toks, ref_logits, ref_ids = [1], [], []
        if self.rank == 0:
            one = Decoder(self.shape, full, stream=self.stream.cuda_stream, numerics="exact")
            tok = 1
            for pos in range(steps):
                nxt = one.step(tok, pos)
                ref_logits.append(one.logits()); ref_ids.append(nxt)
                tok = nxt
                toks.append(tok)
            one.close()
            del one
        box = [toks]
        dist.broadcast_object_list(box, src=0)
        toks = box[0]
        worst, ids_ok = 0.0, True
        self.barrier()
        for pos in range(steps):
            nxt = self.dec.step(toks[pos], pos)
            if self.rank == 0:
                lg = self.dec.logits()
                worst = max(worst, float(np.abs(lg - ref_logits[pos]).max()))
                top2 = np.sort(ref_logits[pos])[-2:]
                if top2[1] - top2[0] > 2 * tol and nxt != ref_ids[pos]:
                    ids_ok = False
        res = {"checked_against": "unsharded single-GPU decoder in exact (bit-identical-to-reference) numerics, same weights, "
                                  "teacher-forced", "numerics": self.numerics, "steps": steps,
               "max_abs_logit_diff": worst, "tolerance": tol, "ids_equal_where_margin_gt_2e-4": ids_ok}
        if self.rank == 0 and (worst > tol or not ids_ok):
            raise SystemExit(f"tensor-parallel decode differs from the unsharded decoder: {res}")
        return res

    # -- measurement ---------------------------------------------------------------------------
    def prepass(self):
        """Untimed: decode 0..CONTEXT-1 (KV cache for every window, warm-up, parity record)."""
        self.barrier()
        n = min(max(CONTEXT, self.args.steps), self.shape.seq_len)
        self.ids = self.dec.generate(1, 0, n)
        again = self.dec.generate(1, 0, min(64, n))
        if again != self.ids[:len(again)]:
            raise SystemExit("decode is not deterministic")
        self.barrier()

    def first_token(self, pos):
        return 1 if pos == 0 else self.ids[pos - 1]

    def _max_over_ranks(self, values):
        if self.world == 1:
            return values
        import torch.distributed as dist
        t = self.torch.tensor(values, device="cuda", dtype=self.torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()

    def time_windows(self, windows, e2e=False):
        """Per-window device time (ms) of one pass over `windows`; max over ranks.  No host work
        between the barrier that aligns the ranks and the opening event."""
        torch = self.torch
        out = []
        for start, n in windows:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            tok = self.first_token(start)
            self.barrier()
            e0.record(self.stream)
            if e2e:
                got = []
                for pos in range(start, start + n):
                    tok = self.dec.step(tok, pos)
                    got.append(tok)
            else:
                got = self.dec.generate(tok, start, n)
            e1.record(self.stream)
            torch.cuda.synchronize()
            if got != self.ids[start:start + n]:
                raise SystemExit(f"window at position {start} ({'e2e' if e2e else 'device loop'}) produced token ids "
                                 "that differ from the pre-pass")
            self.last_ids = got
            out.append(e0.elapsed_time(e1))
        return self._max_over_ranks(out)

    def run(self):
        args, shape = self.args, self.shape
        K = args.steps
        ctx = min(CONTEXT, shape.seq_len)
        windows = plan_windows(K, ctx)
        self.prepass()
        sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", 0))).start() if self.rank == 0 else None
        time.sleep(0.3 if sampler else 0.0)
        reps = max(1, args.reps)
        launches0 = self.lib.kllm_launch_count()
        t_wall0 = time.time()
        totals, per_window = [], []
        for _ in range(reps):
            ms = self.time_windows(windows)
            totals.append(sum(ms)); per_window.append(ms)
        t_wall1 = time.time()
        if args.dump_outputs:
            # what a caller of the timed path holds after its last step (read outside the timed region)
            import numpy as np
            self.last_step = {"logits": self.dec.logits(), "next_token": np.array([self.last_ids[-1]], np.float64)}
        launches = (self.lib.kllm_launch_count() - launches0) // reps
        clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
        ms_total = statistics.median(totals)
        med_rep = per_window[totals.index(sorted(totals)[len(totals) // 2])]

        e2e_reps = max(1, min(reps, 3))
        launches_e0 = self.lib.kllm_launch_count()
        e2e_totals = [sum(self.time_windows(windows, e2e=True)) for _ in range(e2e_reps)]
        launches_e2e = (self.lib.kllm_launch_count() - launches_e0) // e2e_reps
        ms_e2e = statistics.median(e2e_totals)

        by_pos = {}
        for p in (1, 256, 1023):
            if p + 8 <= shape.seq_len and p < len(self.ids):
                n = min(8, len(self.ids) - p)
                t = [self.time_windows([(p, n)])[0] for _ in range(3)]
                by_pos[str(p)] = n / (statistics.median(t) / 1e3)

        from kuiperllama_b200.tensor_parallel import weight_bytes_per_token_per_gpu
        bytes_tok = shape.weight_bytes_per_token()
        bytes_gpu = weight_bytes_per_token_per_gpu(shape, self.world, self.rank, self.dec.classifier_rows)
        peak, peak_src = measured_peaks()
        tok_s = K / (ms_total / 1e3)
        res = {
            "value": tok_s, "ms_per_step": ms_total / K, "steps": K,
            "e2e": {"value": K / (ms_e2e / 1e3), "unit": "tokens/s", "h2d_bytes_per_step": 16, "d2h_bytes_per_step": 16,
                    "reps": e2e_reps},
            "by_position_tok_s": by_pos, "windows": [[s, n] for s, n in windows],
            "rep_totals_ms": totals, "gpu_launches": int(launches), "gpu_launches_e2e": int(launches_e2e),
            "clocks": clocks, "bytes_tok": bytes_tok, "bytes_gpu": bytes_gpu, "classifier_rows": self.dec.classifier_rows,
        }
        if self.engine == "persistent":
            # ONE launch of the persistent megakernel per window: the dominant (only) kernel.  Algorithmic
            # bytes per launch = positions in the window x this GPU's weight bytes per token; duration = the
            # events around that launch (state upload 16 B + kernel + id readback on the same stream).
            n_launch = len(windows)
            ach = bytes_gpu * K / (ms_total / 1e3) / 1e9
            key = "megakernel" if self.world == 1 else f"megakernel_tp{self.world}"
            traffic = ncu_traffic(self.workload, key)
            res["roofline"] = {
                "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": traffic["dram_bytes_per_token"] * K / n_launch if traffic else None,
                "kernel": "decode_megakernel (persistent: whole forward + argmax, %s positions per launch)" %
                          "/".join(sorted({str(n) for _, n in windows})),
                "algorithmic_bytes_per_launch": bytes_gpu * K / n_launch, "avg_launch_us": ms_total * 1e3 / n_launch,
                "launches_timed": n_launch, "peak_source": peak_src, "per_gpu": self.world > 1,
                "traffic_source": traffic}
        else:
            res["roofline"] = {"bound": "hbm", "achieved": bytes_gpu * tok_s / 1e9, "peak": peak, "unit": "GB/s",
                               "frac": bytes_gpu * tok_s / 1e9 / peak, "traffic": None,
                               "kernel": "graph engine: whole decode step (all launches)", "peak_source": peak_src}
        res["median_rep_window_ms"] = med_rep
        return res

    def close(self):
        self.dec.close()
        if self.comm:
            self.comm.close()  # collective (barrier)


def run_ours(args, rank, world):
    import torch
    from kuiperllama_b200 import SHAPES, load_library

    lib = load_library()
    local_rank = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if args.warmup + 1 > CONTEXT:
        raise SystemExit("--warmup exceeds the context")
    stream = torch.cuda.Stream()  # a real stream: the events and the decoder's work share it
    torch.cuda.set_stream(stream)

    b = Bench(args, rank, world, args.workload, stream, lib)
    shape = b.shape
    res = b.run()
    if rank == 0 and args.dump_outputs:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in b.last_step.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)
    line = None
    if rank == 0:
        line = {
            "metric": METRIC, "value": res["value"], "unit": "tokens/s", "n_gpus": world, "steps": res["steps"],
            "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": vs_baseline(args.workload, res["value"]),
            "dtype": "f32" if shape.group_size == 0 else "int8w/f32",
            "data": "synthetic random-init weights (tools/model.py init, seed %d), greedy decode from token 1" % b.seed,
            "config": {"workload": WORKLOAD_NAMES[args.workload], "shape": shape.name,
                       "context": f"1->{min(CONTEXT, shape.seq_len)}: KV cache filled by an untimed pre-pass of "
                                  f"{min(CONTEXT, shape.seq_len)} positions (>= --warmup), then {res['steps']} timed positions in windows [start, n] = "
                                  f"{res['windows']}", "batch": 1,
                       "reps": args.reps, "reported": "median repetition; per window CUDA events on the decoder's stream, max over ranks",
                       "parallelism": "single GPU" if world == 1 else f"tp{world}",
                       "l2": "no flush: every step streams %.2f GB of weights per GPU >> 126 MB L2" % (res["bytes_gpu"] / 1e9),
                       "weight_bytes_per_token": res["bytes_tok"], "launches_per_step": b.launches_per_step,
                       "engine": b.engine,
                       "numerics": "fast: free summation order (int8 rows as int8 weights x 24-bit fixed-point activations on mma.sync s8 / dp4a, "
                                   "flash-decoding attention), logits within 1e-4 of the exact mode "
                                   "(tests/test_decoder_gpu.py::test_fast_numerics_within_north_star_tolerance); "
                                   "exact-mode numbers under \"exact\"" if b.numerics == "fast" else
                                   "exact: every reduction in the reference's order, logits bit-identical to the reference's CUDA path"},
            "e2e": res["e2e"],
            "by_position_tok_s": res["by_position_tok_s"],
            # kernels of libkllm_b200 launched inside ONE repetition of the timed region: the persistent
            # engine decodes a whole window per cooperative launch; the e2e region launches once per token
            "gpu_launches": res["gpu_launches"], "gpu_launches_e2e": res["gpu_launches_e2e"],
            "clocks": res["clocks"], "roofline": res["roofline"],
            "rep_totals_ms": res["rep_totals_ms"],
        }
        if world > 1:
            line["config"]["tp_comm"] = b.comm.backend
            line["config"]["weight_bytes_per_token_per_gpu"] = res["bytes_gpu"]
            line["config"]["classifier_rows_per_gpu"] = res["classifier_rows"]
            line["parity"] = b.parity
    w_cpu = b.w if (world == 1 and not args.no_cpu_baseline) else None
    primary_numerics = b.numerics
    b.close()
    del b
    torch.cuda.empty_cache()

    if primary_numerics == "fast" and not args.no_exact:
        # the verification mode on the same workload: bit-identical to the reference, reported next to the headline
        xargs = argparse.Namespace(**{**vars(args), "reps": min(args.reps, 3)})
        xb = Bench(xargs, rank, world, args.workload, stream, lib, numerics="exact")
        xres = xb.run()
        if rank == 0:
            line["exact"] = {"value": xres["value"], "unit": "tokens/s", "ms_per_step": xres["ms_per_step"],
                             "e2e": xres["e2e"], "by_position_tok_s": xres["by_position_tok_s"],
                             "roofline_frac": xres["roofline"]["frac"], "parity": xb.parity}
        xb.close()
        del xb
        torch.cuda.empty_cache()

    if world > 1 and not args.no_secondary and args.workload != "llama2-7b":
        # BASELINE.json configs[4]: the fp32 Llama-2-7B under the same tensor parallelism
        sargs = argparse.Namespace(**{**vars(args), "reps": min(args.reps, 3)})
        sb = Bench(sargs, rank, world, "llama2-7b", stream, lib)
        sres = sb.run()
        if rank == 0:
            line["secondary"] = {
                "workload": WORKLOAD_NAMES["llama2-7b"], "value": sres["value"], "unit": "tokens/s",
                "ms_per_step": sres["ms_per_step"], "steps": sres["steps"], "e2e": sres["e2e"],
                "by_position_tok_s": sres["by_position_tok_s"], "roofline": sres["roofline"], "parity": sb.parity,
                "weight_bytes_per_token_per_gpu": sres["bytes_gpu"], "windows": sres["windows"]}
        sb.close()
        del sb
    if rank == 0 and w_cpu is not None:
        line["cpu_baseline"] = cpu_reference_run(shape, w_cpu, 256, args.cpu_seconds)
    if rank == 0:
        emit(line)
    if world > 1:
        _leave_process_group()


def main():
    args = parse_args()
    if args.steps < 1:
        raise SystemExit("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        raise SystemExit("--dump-outputs applies to --impl ours")
    # ONE JSON line on stdout: libraries that chat on fd 1 (NCCL prints its version there) go to stderr
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if world == 1 and args.gpus > 1 and args.impl == "ours":
        # plain `python bench.py --gpus N`: become the torchrun launch
        os.execv(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                                  f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
                                  "--master-port", os.environ.get("MASTER_PORT", "29517"),
                                  str(Path(__file__).resolve()), *sys.argv[1:]])
    if args.workload is None:
        args.workload = default_workload(args.gpus)
    if args.seed is None:
        args.seed = SEEDS.get(args.workload, 1234)
    from kuiperllama_b200 import SHAPES
    if args.impl == "ours" and args.steps > SHAPES[args.workload].seq_len:
        raise SystemExit(f"--steps {args.steps} exceeds the context of {SHAPES[args.workload].name} "
                         f"({SHAPES[args.workload].seq_len} positions)")
    if args.impl == "reference":
        run_reference(args, rank, world)
    elif args.impl == "reference-cuda":
        run_reference_cuda(args, rank, world)
    else:
        run_ours(args, rank, world)


if __name__ == "__main__":
    main()
