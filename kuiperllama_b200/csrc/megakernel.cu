// Persistent decode megakernel for sm_100a: the whole per-token forward of LLama2Model /
// Qwen2Model (kuiper/source/model/llama3.cpp:147-167, 600-745) in ONE cooperative launch that
// can run any number of consecutive positions.
//
// Why: at batch 1 the path is a 4-26 GB/token weight stream; with one launch per op (even 6
// fused launches per layer in a CUDA graph) every kernel boundary drains the HBM pipeline
// (profiles/r01a: 15-42 % DRAM utilisation per kernel).  Here one CTA per SM stays resident
// and a dedicated producer warp streams that CTA's share of EVERY weight matrix, in schedule
// order, through a ring of shared-memory stages with TMA bulk copies (cp.async.bulk ->
// UBLKCP) signalled on mbarriers.  Weights never depend on activations, so the producer runs
// ahead across every dependency of the token; a second producer warp walks the same schedule a
// few stages further ahead and only pulls the bytes into L2 (cp.async.bulk.prefetch.L2), so
// HBM keeps fetching while SMs wait for each other.
//
// Schedule per layer:  QKV(+bias) | attention(+RoPE) | Wo | W1,W3->SiLU*gate | W2 ; then
// classifier + greedy argmax.  RoPE moves into the attention phase so GEMV rows can be split
// evenly over all SMs.
//
// Consumers (CW warps: 8 for fp32 weights, 14 for int8): the rows of a ring stage are handed out as TASKS of
// up to four rows to one warp each, round-robin.  A task's rows share every load of the input vector, their
// dot-product chains interleave (ILP instead of occupancy), their totals are folded with "packed" shuffle trees
// (kllm_device.cuh) that do the additions of cub's tree only, and one lane per row runs the epilogues side by
// side.  (int8, toleranced mode, opt-in: a team of warps shares a stage -- mma.sync s8 or dp4a; gemv_phase.)
//
// No local memory: the ring takes the whole unified L1, so a stack access is a round trip to L2.  The kernel
// parameters are __grid_constant__ (never copied to the stack), register buffers are always written in full
// (a conditionally written element forces the array into local memory), nothing indexes an array at run time.
// `cuobjdump -res-usage` / tools/sass_histogram.py (profiles/r02_sass_histogram.txt) show what is left.
//
// Hand-over between phases (KLLM_MEGA_TAGGED=2, default): every produced element is published as
// one 64-bit {tag, fp32} word and polled in place by the consuming phase -- no fences, flags or
// grid barriers; the residual-stream update after Wo and W2 is summed by the reader
// (x = x_old + sum over ranks, x_old living in the CTA's own shared memory), which under tensor
// parallelism makes the same stores, sent to every rank over NVLink peer mappings, the
// all-reduce.  One grid barrier per token remains (before the argmax fold).  KLLM_MEGA_TAGGED=1
// keeps grid barriers for the hand-offs inside a layer, 0 uses grid barriers everywhere (single
// GPU only).
//
// Arithmetic is the same as the per-op kernels (gemv.cu / attention.cu / elementwise.cu): every
// dot product, reduction tree, softmax sum and value chain reproduces the reference CUDA
// kernels' floating-point order, so logits stay bit-identical to the reference's CUDA path.
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include <cfloat>
#include <cstdint>
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "../../include/kllm_b200.h"
#include "kllm_device.cuh"
#include "kllm_host.h"
#include "megakernel.h"

namespace kllm {
namespace mega {

// The phase bodies are written as functions but inlined: real calls make ptxas spill around them,
// and with the ring taking all of shared memory there is no L1 left -- a spill is an L2 round trip.
#ifndef KLLM_MBAR_HINT_NS
#define KLLM_MBAR_HINT_NS 20000u
#endif
// 1: warps without a row in an attention tile skip its wait and block at a hardware barrier instead of
// spinning on the mbarrier.  Measured on B200 (profiles/README.md, pass M): no gain (826 vs 837 tok/s), so off.
#ifndef KLLM_ATTN_GATE
#define KLLM_ATTN_GATE 0
#endif
#ifndef KLLM_TASK_ROWS
#define KLLM_TASK_ROWS 4
#endif
#ifndef KLLM_PHASE_CALL
#define KLLM_PHASE_CALL __forceinline__
#endif
#ifndef KLLM_STAGE_CALL
#define KLLM_STAGE_CALL __noinline__  // once per phase, and their poll buffers would otherwise push the row loops' state out
#endif
constexpr int kMaxStages = 16;
constexpr int kMaxWarps = 16;
constexpr int kSoftmaxThreads = 256;  // mha_kernel.cu:112-127 launches 256 threads per head
constexpr int kNormThreads = 128;     // rmsnorm_kernel.cu:58-77 launches 128 threads
constexpr long long kSpinLimit = 120000000000LL;  // ~1 minute of SM clocks: a lost peer becomes a trap

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* b, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* b, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* b) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory");
}
// try_wait suspends the warp in hardware until the phase completes or the time hint (ns) runs out:
// with a generous hint a waiting warp sleeps instead of re-issuing the probe -- waiting warps
// otherwise compete for issue slots with the warps that are computing on the same scheduler
// (ncu, r02f: SYNCS + BRA + YIELD of the spin loops were a quarter of all executed instructions).
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity) {
  asm volatile(
      "{\n .reg .pred p;\n WAIT_%=:\n"
      " mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
      " @p bra DONE_%=;\n bra WAIT_%=;\n DONE_%=:\n}" ::"r"(smem_u32(b)),
      "r"(parity), "r"(KLLM_MBAR_HINT_NS)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar,
                                         uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
      "[%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}
__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
// Non-blocking "pull this span into L2": no shared memory, no completion to wait for.
__device__ __forceinline__ void bulk_prefetch_l2(const void* src, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ uint64_t policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_add(unsigned* p, unsigned v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// 64-bit {tag, value} words of the tagged exchange: single-copy atomic, so value and tag travel
// together and no fence or flag is needed between a writer on one GPU and a reader on another.
__device__ __forceinline__ unsigned long long tagged_word(float v, unsigned tag) {
  return (static_cast<unsigned long long>(tag) << 32) | __float_as_uint(v);
}
__device__ __forceinline__ void st_tagged(unsigned long long* p, float v, unsigned tag) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(tagged_word(v, tag)) : "memory");
}
__device__ __forceinline__ void ld_tagged2(const unsigned long long* p, unsigned long long& a,
                                           unsigned long long& b) {
  asm volatile("ld.relaxed.sys.global.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}
// local (same GPU) flavour of the tagged words
__device__ __forceinline__ void st_tagged_gpu(unsigned long long* p, float v, unsigned tag) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(tagged_word(v, tag)) : "memory");
}
__device__ __forceinline__ void st_tagged2_gpu(unsigned long long* p, float v0, float v1, unsigned tag) {  // 16-byte aligned
  asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(tagged_word(v0, tag)), "l"(tagged_word(v1, tag))
               : "memory");
}
__device__ __forceinline__ unsigned long long ld_tagged_gpu(const unsigned long long* p) {
  unsigned long long w;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(w) : "l"(p) : "memory");
  return w;
}
__device__ __forceinline__ void ld_tagged2_gpu(const unsigned long long* p, unsigned long long& a,
                                               unsigned long long& b) {
  asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}
__device__ __forceinline__ unsigned tag_of(unsigned long long w) { return static_cast<unsigned>(w >> 32); }
__device__ __forceinline__ float val_of(unsigned long long w) { return __uint_as_float(static_cast<unsigned>(w)); }

// A polled word may carry an OLDER tag (its producer is still on its way) but never a NEWER one:
// the slot-reuse argument (megakernel.h) says nobody publishes use n+1 of a word before everybody
// consumed use n.  A newer tag is therefore a protocol error and traps at once; a word that never
// turns up becomes a trap after a bounded spin, not a hang.
__device__ __noinline__ void poll_failed(unsigned seen, unsigned want, long long t_start, int what) {
  const char* name = what == 0 ? "hand-off word" : (what == 1 ? "residual exchange" : "phase input");
  if (static_cast<int>(seen - want) > 0) {
    printf("kllm mega: cta %d thread %d: %s carries tag %u, newer than the awaited %u (protocol error)\n",
           blockIdx.x, threadIdx.x, name, seen, want);
    __trap();
  }
  if (clock64() - t_start > kSpinLimit) {
    printf("kllm mega: cta %d thread %d timed out on %s tag %u (last seen %u)\n", blockIdx.x, threadIdx.x,
           name, want, seen);
    __trap();
  }
}
__device__ __forceinline__ unsigned long long ld_tagged_sys(const unsigned long long* p) {
  unsigned long long w;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(w) : "l"(p) : "memory");
  return w;
}
// spin until the word (written by any rank) carries `tag`
__device__ __forceinline__ float poll_tagged_sys(const unsigned long long* p, unsigned tag) {
  unsigned long long w = ld_tagged_sys(p);
  if (tag_of(w) != tag) {
    const long long t0 = clock64();
    do {
      poll_failed(tag_of(w), tag, t0, 1);
      w = ld_tagged_sys(p);
    } while (tag_of(w) != tag);
  }
  return val_of(w);
}
// spin until the word carries `tag`
__device__ __forceinline__ float poll_tagged(const unsigned long long* p, unsigned tag) {
  unsigned long long w = ld_tagged_gpu(p);
  if (tag_of(w) != tag) {
    const long long t0 = clock64();
    do {
      poll_failed(tag_of(w), tag, t0, 0);
      w = ld_tagged_gpu(p);
    } while (tag_of(w) != tag);
  }
  return val_of(w);
}
template <int CT>
__device__ __forceinline__ void consumer_sync() {
  asm volatile("bar.sync 1, %0;" ::"n"(CT) : "memory");
}

__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

struct Pipe {
  int slot;
  uint32_t parity;
  __device__ __forceinline__ void advance(int stages) {
    if (++slot == stages) {
      slot = 0;
      parity ^= 1u;
    }
  }
};

// Static shared memory (namespace scope, so the phase functions address it with immediates instead of
// pointers held in registers).  The ring leaves only a few KB of L1, so everything the inner loops
// touch lives in shared memory or registers: the schedule entries the consumers, the ring producer
// and the L2 prefetcher are working on (usually three different phases), the barriers and the
// reduction scratch.
__shared__ uint64_t g_full_bar[kMaxStages];
__shared__ uint64_t g_empty_bar[kMaxStages];
__shared__ float g_s_warp[kMaxWarps];
__shared__ float g_s_argv[kMaxWarps];
__shared__ int g_s_argi[kMaxWarps];
__shared__ float g_s_bcast;
__shared__ volatile unsigned g_fill_count;  // ring stages the producer has issued so far
__shared__ float g_s_team[kMaxWarps / 2][2][3][8];  // team form: the other members' row partials, double buffered per team
__shared__ Phase g_ph_cons;
__shared__ Phase g_ph_prod;
__shared__ Phase g_ph_pf;
constexpr int kCtlBytes = 0;
extern __shared__ __align__(128) unsigned char smem[];
// per-thread state the phase functions hand back to the kernel loop
struct Carry {
  Pipe pipe;
  float best_v;
  int best_i;
};

// Grid barrier over the consumer threads of all CTAs.  Monotonic counter, wrap-safe compare.
template <int CT>
__device__ __forceinline__ void grid_barrier(unsigned* counter, unsigned& target, unsigned grid) {
  consumer_sync<CT>();
  target += grid;
  if (threadIdx.x == 0) {
    red_release_add(counter, 1u);
    while (static_cast<int>(ld_acquire_u32(counter) - target) < 0) {
    }
  }
  consumer_sync<CT>();
}

// ---- unit -> (segment, row) ------------------------------------------------------------------
struct RowRef {
  int seg;
  int row;
};
__device__ __forceinline__ RowRef resolve_row(const Phase& ph, int unit, int sub) {
  if (ph.swiglu) return RowRef{sub, unit};
  int seg = 0, row = unit;
  if (ph.n_seg > 1 && row >= ph.seg[0].rows) {
    row -= ph.seg[0].rows;
    seg = 1;
    if (ph.n_seg > 2 && row >= ph.seg[1].rows) {
      row -= ph.seg[1].rows;
      seg = 2;
    }
  }
  return RowRef{seg, row};
}

// Row j of a ring stage that starts at unit u and holds n units, in STAGE ORDER.  SwiGLU stages
// keep their w1 rows first and their w3 rows after them, so that each half -- like any run of
// consecutive rows of one matrix -- is ONE contiguous span of the checkpoint and one bulk copy.
__device__ __forceinline__ RowRef stage_row(const Phase& ph, int u, int n, int j) {
  if (ph.swiglu) return j < n ? RowRef{0, u + j} : RowRef{1, u + j - n};
  return resolve_row(ph, u + j, 0);
}
// Lane j (< nrows) holds row j of the stage: returns the length of the run of consecutive rows
// of one matrix that STARTS at this lane (0 for lanes inside a run).
__device__ __forceinline__ int run_length(const RowRef& rr, int lane, int nrows) {
  const int pseg = __shfl_up_sync(kFull, rr.seg, 1);
  const int prow = __shfl_up_sync(kFull, rr.row, 1);
  const bool head = lane < nrows && (lane == 0 || rr.seg != pseg || rr.row != prow + 1);
  const unsigned heads = __ballot_sync(kFull, head);
  if (!head) return 0;
  const unsigned later = heads & ~((2u << lane) - 1u);
  return (later ? __ffs(later) - 1 : nrows) - lane;
}

// ---- exact-order accumulation from shared memory ----------------------------------------------
// The row loops address shared memory by 32-bit shared-window addresses through explicit
// ld.shared: behind the call boundary of dot_rows the compiler no longer knows the pointers are
// shared memory (it would emit generic loads), and `volatile` keeps the loads in program order --
// a batch of loads first, then the math that consumes them.
__device__ __forceinline__ float4 lds_f4(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ float lds_f32(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
  return v;
}

// fp32: virtual thread (lane + 32 j) owns packs base + 32 j + lane (matmul_kernel.cu:27-35).  The
// NR rows of a task share each load of x; per batch (two 32-pack columns) 2 x loads and 2 NR weight
// loads are issued before the 2 NR independent dot4 chains.
template <int NR>
__device__ __forceinline__ void accum_f32(const uint32_t (&w)[NR], uint32_t x, int n_packs, int lane,
                                          float (&acc)[NR][4]) {
  // Full 128-pack blocks run branch-free with all 4 * (1 + NR) shared loads issued before the math
  // (two blocks in flight), so the four independent chains per row overlap the LDS latency.
  const int full = n_packs & ~127;
  uint32_t xp = x + lane * 16;
  uint32_t wp[NR];
#pragma unroll
  for (int r = 0; r < NR; ++r) wp[r] = w[r] + lane * 16;
#pragma unroll 2
  for (int base = 0; base < full; base += 128) {
    float4 xv[4];
    float4 wv[NR][4];
#pragma unroll
    for (int j = 0; j < 4; ++j) xv[j] = lds_f4(xp + 512 * j);
#pragma unroll
    for (int r = 0; r < NR; ++r)
#pragma unroll
      for (int j = 0; j < 4; ++j) wv[r][j] = lds_f4(wp[r] + 512 * j);
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int r = 0; r < NR; ++r) acc[r][j] = __fadd_rn(dot4_ref(xv[j], wv[r][j]), acc[r][j]);
    xp += 2048;
#pragma unroll
    for (int r = 0; r < NR; ++r) wp[r] += 2048;
  }
  if (full < n_packs) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (full + 32 * j + lane < n_packs) {
        const float4 xv = lds_f4(xp + 512 * j);
#pragma unroll
        for (int r = 0; r < NR; ++r) acc[r][j] = __fadd_rn(dot4_ref(xv, lds_f4(wp[r] + 512 * j)), acc[r][j]);
      }
    }
  }
}

// int8, group size 64 (export.py --version 3): virtual thread (4 lane + e) owns elements
// 128 k + 4 lane + e (matmul_kernel.cu:70-74), so the lane's four bytes of chunk k sit in group
// 2 k + (lane >> 4) of the row: the scale address just steps by two floats.  Per element the
// reference's fma(x * scale, float(w), acc) -- PRMT + FADD (exact int8 -> fp32) + FMUL + FFMA;
// everything else (one 4-byte weight load and one scale load per row, one 16-byte x load per chunk,
// the xor that prepares the byte permutes) is shared by four elements or by the NR rows.  Chunk
// k + 1 is loaded while chunk k is computed.
// `sc[r]`: the row's staged scales (rows start on a group boundary -- checked on the host).
template <int NR>
__device__ __forceinline__ void accum_w8_g64(const uint32_t (&w)[NR], const uint32_t (&sc)[NR], uint32_t x,
                                             int M, int lane, float (&acc)[NR][4]) {
  const int chunks = M >> 7;
  const bool tail = (chunks << 7) + (lane << 2) < M;  // M % 128 != 0: a last, partial chunk
  const int total = chunks + (tail ? 1 : 0);
  if (total == 0) return;
  uint32_t xp = x + lane * 16;
  uint32_t wp[NR], sp[NR];
#pragma unroll
  for (int r = 0; r < NR; ++r) {
    wp[r] = w[r] + lane * 4;
    sp[r] = sc[r] + (lane >> 4) * 4;
  }
  float4 xv = lds_f4(xp);
  uint32_t packed[NR];
  float s[NR];
#pragma unroll
  for (int r = 0; r < NR; ++r) {
    packed[r] = lds_u32(wp[r]);
    s[r] = lds_f32(sp[r]);
  }
#pragma unroll 2
  for (int k = 0; k < total; ++k) {
    if (k + 1 < total) {  // uniform per virtual-thread quad: lanes past a partial tail chunk have total == chunks
      xp += 512;
#pragma unroll
      for (int r = 0; r < NR; ++r) {
        wp[r] += 128;
        sp[r] += 8;
      }
    }
    const float4 xn = lds_f4(xp);  // last iteration: re-reads its own chunk (harmless)
    uint32_t pn[NR];
    float sn[NR];
#pragma unroll
    for (int r = 0; r < NR; ++r) {
      pn[r] = lds_u32(wp[r]);
      sn[r] = lds_f32(sp[r]);
    }
#pragma unroll
    for (int r = 0; r < NR; ++r) {
      float wf[4];
      int8x4_to_float(packed[r], wf);
      acc[r][0] = __fmaf_rn(__fmul_rn(xv.x, s[r]), wf[0], acc[r][0]);
      acc[r][1] = __fmaf_rn(__fmul_rn(xv.y, s[r]), wf[1], acc[r][1]);
      acc[r][2] = __fmaf_rn(__fmul_rn(xv.z, s[r]), wf[2], acc[r][2]);
      acc[r][3] = __fmaf_rn(__fmul_rn(xv.w, s[r]), wf[3], acc[r][3]);
    }
    xv = xn;
#pragma unroll
    for (int r = 0; r < NR; ++r) {
      packed[r] = pn[r];
      s[r] = sn[r];
    }
  }
}

// int8, any other group size (multiple of 4): the group index is computed per chunk.
template <int NR>
__device__ __forceinline__ void accum_w8_any(const uint32_t (&w)[NR], const uint32_t (&sc)[NR], uint32_t x,
                                             int M, int group_shift, int group_size, int lane,
                                             float (&acc)[NR][4]) {
  const int full_chunks = M >> 7;
  auto one = [&](int k) {
    const int i = (k << 7) + (lane << 2);
    const float4 xv = lds_f4(x + i * 4);
    const int g = group_shift >= 0 ? (i >> group_shift) : (i / group_size);
#pragma unroll
    for (int r = 0; r < NR; ++r) {
      const uint32_t packed = lds_u32(w[r] + i);
      const float s = lds_f32(sc[r] + g * 4);
      float wf[4];
      int8x4_to_float(packed, wf);
      acc[r][0] = __fmaf_rn(__fmul_rn(xv.x, s), wf[0], acc[r][0]);
      acc[r][1] = __fmaf_rn(__fmul_rn(xv.y, s), wf[1], acc[r][1]);
      acc[r][2] = __fmaf_rn(__fmul_rn(xv.z, s), wf[2], acc[r][2]);
      acc[r][3] = __fmaf_rn(__fmul_rn(xv.w, s), wf[3], acc[r][3]);
    }
  };
#pragma unroll 2
  for (int k = 0; k < full_chunks; ++k) one(k);
  if ((full_chunks << 7) + (lane << 2) < M) one(full_chunks);
}

// ---- int8 weights x fixed-point activations on the integer dot-product unit (TOLERANCED) ---------
// The exact int8 loop above is bound by instruction issue: four instructions per weight byte
// (PRMT + FADD to convert, FMUL by the group scale, FFMA), ~21 warp instructions per 128 weight
// bytes against ~5.6 bytes per clock per scheduler that HBM can deliver.  The fast mode turns the
// activations of each 64-element group into 24-bit fixed point once per phase --
//     x_i ~= step_g * q_i,  q_i = round(x_i / step_g),  step_g = max|x in group| / 2^22,
// q_i split into three balanced base-256 digits l2 l1 l0 (int8 each) -- and then needs ONE dp4a per
// 4 weights and digit: sum_i w_i x_i = s_g * step_g * (65536 D2 + 256 D1 + D0), D_k = sum_i w_i l_k,i
// exact in int32.  ~6 warp instructions per 128 weight bytes.  The group scale s_g and the int8
// weights enter exactly as in the reference (dequantised weight = q * s, export.py:60-67); only x is
// rounded, to 2^-23 of its group maximum -- the same order as fp32 rounding of the products
// themselves.  Logits agree with the exact mode to ~1e-6 relative (tests: <= 1e-4 absolute, same
// greedy id wherever the top-2 margin exceeds 2e-4), not bit for bit.
__device__ __forceinline__ uint4 lds_u4(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ int dp4a4(const uint4& w, const uint4& l) {
  int d = __dp4a(static_cast<int>(w.x), static_cast<int>(l.x), 0);
  d = __dp4a(static_cast<int>(w.y), static_cast<int>(l.y), d);
  d = __dp4a(static_cast<int>(w.z), static_cast<int>(l.z), d);
  return __dp4a(static_cast<int>(w.w), static_cast<int>(l.w), d);
}
// exact int32 -> fp32 for |d| < 2^22 without the slow conversion pipe: 1.5 * 2^23 + d is exact
__device__ __forceinline__ float small_int_to_float(int d) {
  return __fsub_rn(__int_as_float(0x4B400000 + d), 12582912.0f);
}
// In-place layout (fast mode): the 256 bytes that held the fp32 values of 64-element group g hold four
// 64-byte regions -- the three digit planes of the group and its step.  Digit plane k sits in region
// (k + (g & 1)) & 3, the step in region (3 + (g & 1)) & 3: alternating the region order between even
// and odd groups makes the 32 lanes of a 128-bit load (8 groups x 4 quarters) hit all 8 distinct
// 16-byte bank slots, 4 lanes each -- the minimum of 4 wavefronts.  Quarter q (16 elements) of a
// plane is the 16-byte chunk q of its region.
template <int NR>
__device__ __forceinline__ void accum_w8_dp4a(const uint32_t (&w)[NR], const uint32_t (&sc)[NR], uint32_t x, int M,
                                              int lane, float (&acc)[NR], int it_begin = 0, int it_end = 1 << 30) {
  // lane owns 16 consecutive elements per step of 512: group = 8 * step + lane / 4, quarter = lane % 4
  const uint32_t odd = (lane >> 2) & 1u;
  const uint32_t gq = x + (lane >> 2) * 256 + (lane & 3) * 16;
  const uint32_t l0 = gq + ((0u + odd) & 3u) * 64, l1 = gq + ((1u + odd) & 3u) * 64, l2 = gq + ((2u + odd) & 3u) * 64;
  const uint32_t xsp = x + (lane >> 2) * 256 + ((3u + odd) & 3u) * 64;
  uint32_t wp[NR], sp[NR];
#pragma unroll
  for (int r = 0; r < NR; ++r) {
    wp[r] = w[r] + lane * 16;
    sp[r] = sc[r] + (lane >> 2) * 4;
  }
  const int steps = min((M + 511) >> 9, it_end);
#pragma unroll 2
  for (int it = it_begin; it < steps; ++it) {
    if (it * 512 + lane * 16 < M) {  // M % 512 != 0: the last step covers part of the lanes (M % 64 == 0)
      const uint4 a0 = lds_u4(l0 + it * 2048), a1 = lds_u4(l1 + it * 2048), a2 = lds_u4(l2 + it * 2048);
      const float xstep = lds_f32(xsp + it * 2048);
#pragma unroll
      for (int r = 0; r < NR; ++r) {
        const uint4 wv = lds_u4(wp[r] + it * 512);
        const float ws = lds_f32(sp[r] + it * 32);
        const float c0 = small_int_to_float(dp4a4(wv, a0));
        const float c1 = small_int_to_float(dp4a4(wv, a1));
        const float c2 = small_int_to_float(dp4a4(wv, a2));
        const float f = __fmaf_rn(c2, 65536.0f, __fmaf_rn(c1, 256.0f, c0));
        acc[r] = __fmaf_rn(f, __fmul_rn(xstep, ws), acc[r]);
      }
    }
  }
}

// ---- int8 weights x fixed-point activations on the tensor cores (TOLERANCED, same numbers as above) ----------
// The integer dot-product unit runs at a quarter of the FP32 rate on sm_100 (measured: the dp4a rows above are
// bound by it, 12 IDP.4A per 16 weights), so where a ring stage holds several rows that share the input
// vector -- every matrix with 4096-byte rows -- the 64-element groups go through mma.sync m16n8k32 (s8 x s8 ->
// s32, SASS IMMA.16832.S8.S8) instead:
//     A (16 x 32, row major)  rows 0..7 = the (up to 8) weight rows of the stage, rows 8..15 mirror them
//     B (32 x 8, column major) columns 0, 1, 2 = the three digit planes of x, columns 3..7 = 0
//     D (16 x 8, s32)          D[r][k] = sum_i w[r][i] * l_k[i]  -- the exact integers D_k of the dp4a form
// two mma per group (K = 2 x 32); the lane that holds D[r][0..1] fetches D[r][2] from its neighbour and adds
// s_g * step_g * (65536 D2 + 256 D1 + D0) to the row's running sum.  A PAIR of warps takes a whole stage (the
// ring holds only six stages: one warp per stage would leave most consumer warps idle): the even warp the first
// half of the groups, the odd warp the second half; the halves meet through shared memory.  Rows are
// staged `row_stride` bytes apart = row length + 16, which spreads the eight rows of a fragment load over all
// 32 banks (row r, k-quad t -> bank 4 r + t); the scale rows likewise.
// Result: lane 4 r holds the total of row r (rows >= nrows repeat row nrows - 1).
__device__ __forceinline__ void mma_s8(int (&c)[4], uint32_t a0, uint32_t a2, uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k32.row.col.s32.s8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3])
      : "r"(a0), "r"(a0), "r"(a2), "r"(a2), "r"(b0), "r"(b1));
}
__device__ __forceinline__ float accum_w8_mma(uint32_t w_base, uint32_t row_stride, uint32_t sc_base, uint32_t sc_stride,
                                              int nrows, uint32_t x, int g_begin, int g_end, int lane) {
  const int gid = lane >> 2, tig = lane & 3;
  const int r = min(gid, nrows - 1);
  const uint32_t wrow = w_base + static_cast<uint32_t>(r) * row_stride + static_cast<uint32_t>(tig) * 4u;
  const uint32_t srow = sc_base + static_cast<uint32_t>(r) * sc_stride;
  const uint32_t plane = static_cast<uint32_t>(min(gid, 2));
  const bool bcol = gid < 3;
  float acc = 0.f;
#pragma unroll 2
  for (int g = g_begin; g < g_end; ++g) {
    const uint32_t odd = static_cast<uint32_t>(g) & 1u;
    const uint32_t xg = x + static_cast<uint32_t>(g) * 256u;
    const uint32_t pb = xg + ((plane + odd) & 3u) * 64u + static_cast<uint32_t>(tig) * 4u;
    uint32_t b0 = lds_u32(pb), b1 = lds_u32(pb + 16), b2 = lds_u32(pb + 32), b3 = lds_u32(pb + 48);
    if (!bcol) b0 = b1 = b2 = b3 = 0u;
    const uint32_t wa = wrow + static_cast<uint32_t>(g) * 64u;
    const uint32_t a0 = lds_u32(wa), a1 = lds_u32(wa + 16), a2 = lds_u32(wa + 32), a3 = lds_u32(wa + 48);
    const float xstep = lds_f32(xg + ((3u + odd) & 3u) * 64u);
    const float ws = lds_f32(srow + static_cast<uint32_t>(g) * 4u);
    int c[4] = {0, 0, 0, 0};
    mma_s8(c, a0, a1, b0, b1);  // elements 0..31 of the group
    mma_s8(c, a2, a3, b2, b3);  // elements 32..63
    // c[0] = D[row gid][column 2 tig], c[1] = D[row gid][column 2 tig + 1]: |D| <= 64 * 128 * 128 = 2^20
    const int d2 = __shfl_down_sync(kFull, c[0], 1);  // for the tig == 0 lanes: column 2 lives in tig 1
    const float f = __fmaf_rn(small_int_to_float(d2), 65536.0f,
                              __fmaf_rn(small_int_to_float(c[1]), 256.0f, small_int_to_float(c[0])));
    acc = __fmaf_rn(f, __fmul_rn(xstep, ws), acc);
  }
  return acc;
}

// The phase's input vector (fp32, M floats at xs, M % 64 == 0) -> digit planes + step per group, in
// place (layout above).  Four adjacent lanes share a group: each reads its 16 values, the group
// maximum is folded with two shuffles, and after a warp-level sync (all four have read) each lane
// overwrites its quarter -- no CTA barrier, no values parked in registers.
template <int CT>
__device__ __noinline__ void quantize_input_inplace(float* xs, int M, int tid) {
  const int quarters = M >> 4;
  for (int base = 0; base < quarters; base += CT) {  // CT % 32 == 0: whole warps, groups never straddle one
    const int qg = base + tid;
    const bool on = qg < quarters;
    // lanes past the end read the last quarter again (their group is entirely past the end: M % 64 == 0),
    // so v[] is always written and stays in registers instead of local memory
    float4 v[4];
    float gmax = 0.f;
    {
      const float4* g4 = reinterpret_cast<const float4*>(xs) + min(qg, quarters - 1) * 4;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        v[j] = g4[j];
        gmax = fmaxf(gmax, fmaxf(fmaxf(fabsf(v[j].x), fabsf(v[j].y)), fmaxf(fabsf(v[j].z), fabsf(v[j].w))));
      }
    }
    gmax = fmaxf(gmax, __shfl_xor_sync(kFull, gmax, 1));
    gmax = fmaxf(gmax, __shfl_xor_sync(kFull, gmax, 2));  // also orders: every lane of the group has read
    const float step = w8_group_step(gmax);
    const float inv = w8_group_inv(gmax);
    __syncwarp();
    if (on) {
      const int g = qg >> 2, q = qg & 3;
      const unsigned odd = g & 1;
      unsigned char* gb = reinterpret_cast<unsigned char*>(xs) + g * 256 + q * 16;
      uint32_t* o0 = reinterpret_cast<uint32_t*>(gb + ((0u + odd) & 3u) * 64);
      uint32_t* o1 = reinterpret_cast<uint32_t*>(gb + ((1u + odd) & 3u) * 64);
      uint32_t* o2 = reinterpret_cast<uint32_t*>(gb + ((2u + odd) & 3u) * 64);
#pragma unroll
      for (int j = 0; j < 4; ++j) {  // 4 elements -> one word of each digit plane, written at once
        const float e[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
        uint32_t p0, p1, p2;
        w8_digits4(e, inv, p0, p1, p2);  // kllm_device.cuh: the definition shared with the kind::i8 GEMM
        o0[j] = p0, o1[j] = p1, o2[j] = p2;
      }
      if (q == 0) *reinterpret_cast<float*>(gb + ((3u + odd) & 3u) * 64) = step;
    }
  }
  consumer_sync<CT>();
}

// Dot products of the NR rows of a task (shared-window addresses of the rows and of their int8
// scales); every lane gets every total.  Deliberately NOT inlined: as part of the megakernel's one
// big function the row loops inherit its register pressure and ptxas then serialises every
// shared-memory load with its dependent math; as a function of their own they keep a batch of loads
// in flight.
struct Rows4 {
  uint32_t a[4];
};
template <int NR, bool INT8>
__device__ __forceinline__ float4 dot_rows(Rows4 rows, Rows4 scales, uint32_t x, int M, int group_size,
                                           int group_shift, int lane, bool fast = false) {
  float acc[NR][4];
#pragma unroll
  for (int r = 0; r < NR; ++r)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[r][j] = 0.f;
  float d[4] = {0.f, 0.f, 0.f, 0.f};
  uint32_t w[NR], sc[NR];
#pragma unroll
  for (int r = 0; r < NR; ++r) {
    w[r] = rows.a[r];
    sc[r] = scales.a[r];
  }
  if constexpr (INT8) {
    if (fast) {  // fixed-point activations x int8 weights on dp4a (toleranced mode; group size 64)
      float a1[NR];
#pragma unroll
      for (int r = 0; r < NR; ++r) a1[r] = 0.f;
      accum_w8_dp4a<NR>(w, sc, x, M, lane, a1);
#pragma unroll
      for (int r = 0; r < NR; ++r) {
        float v = a1[r];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(kFull, v, off);
        d[r] = v;
      }
      return make_float4(d[0], d[1], d[2], d[3]);
    }
    if (group_size == 64)
      accum_w8_g64<NR>(w, sc, x, M, lane, acc);
    else
      accum_w8_any<NR>(w, sc, x, M, group_shift, group_size, lane, acc);
#pragma unroll
    for (int r = 0; r < NR; ++r) d[r] = block128_sum_quad_packed(acc[r]);
  } else {
    accum_f32<NR>(w, x, M >> 2, lane, acc);
#pragma unroll
    for (int r = 0; r < NR; ++r) d[r] = block128_sum_vt_packed(acc[r], lane);
  }
  return make_float4(d[0], d[1], d[2], d[3]);
}

struct ArgBest {
  float v;
  int i;
};
__device__ __forceinline__ void arg_fold(ArgBest& a, float ov, int oi) {
  if (oi >= 0 && (a.i < 0 || ov > a.v || (ov == a.v && oi < a.i))) {
    a.v = ov;
    a.i = oi;
  }
}

// (defined below; the P.V phase polls its scores with it)
template <int UP>
__device__ KLLM_STAGE_CALL void stage_handoff(const unsigned long long* src, unsigned tag, int n4, int t, int NT,
                                              float4* xs4);

// ---- inputs of an attention CTA: q (this head), raw k and v (its kv head) of the current position ------------
// Thread i < hs/2 needs its pair of q (and, in the CTA that handles the new key row, of k); thread d < hs the
// value element d.  With tagged hand-offs these are up to five words per thread; polled one after the other
// (each poll a spin loop of its own) they cost five dependent L2 round trips at the head of the layer's
// critical path -- here all of a thread's words are in flight together and re-read together until every tag is
// current.  Slots a thread does not need alias a word it does need.
struct AttnIn {
  float q0, q1, k0, k1, v;
};
__device__ __forceinline__ AttnIn poll_attention_inputs(const unsigned long long* pq0, const unsigned long long* pq1,
                                                        const unsigned long long* pk0, const unsigned long long* pk1,
                                                        const unsigned long long* pv, unsigned tag) {
  unsigned long long w[5];
  w[0] = ld_tagged_gpu(pq0), w[1] = ld_tagged_gpu(pq1), w[2] = ld_tagged_gpu(pk0), w[3] = ld_tagged_gpu(pk1);
  w[4] = ld_tagged_gpu(pv);
  // (no dynamic index into w[]: that would put the buffer into local memory)
  unsigned seen = tag;
  auto stale = [&]() -> bool {
    bool bad = false;
#pragma unroll
    for (int i = 0; i < 5; ++i)
      if (tag_of(w[i]) != tag) bad = true, seen = tag_of(w[i]);
    return bad;
  };
  if (stale()) {
    const long long t0 = clock64();
    do {
      poll_failed(seen, tag, t0, 0);
      w[0] = ld_tagged_gpu(pq0), w[1] = ld_tagged_gpu(pq1), w[2] = ld_tagged_gpu(pk0), w[3] = ld_tagged_gpu(pk1);
      w[4] = ld_tagged_gpu(pv);
    } while (stale());
  }
  return AttnIn{val_of(w[0]), val_of(w[1]), val_of(w[2]), val_of(w[3]), val_of(w[4])};
}

// RoPE on q (this head) and -- with_k -- on the new key row (rope_kernel.cu as compiled, elementwise.cu); the
// rotated key goes to k_s and, by one CTA per kv head, into the cache row of `pos`.  Returns this thread's
// element of the value row (with_v, tid < hs), else 0.  `v_plain`: where thread tid reads its value element when
// the hand-offs are not tagged.
__device__ __forceinline__ float attention_inputs(const Params& P, const Phase& ph, int head, int kvh, int pos, unsigned tag_in,
                                                  bool with_k, bool with_v, float* q_s, float* k_s, float* kcache,
                                                  const float* v_plain) {
  const int tid = threadIdx.x;
  const int hs = P.head_size, seq_len = P.seq_len;
  const bool handoff = ph.tq != nullptr;  // q / k / v arrive as tagged words: no barrier before us
  const bool need_q = tid < hs / 2, need_k = need_q && with_k, need_v = with_v && tid < hs;
  if (!need_q && !need_v) return 0.f;
  int i0, i1;
  if (P.flavour == KLLM_FLAVOUR_LLAMA2) {
    i0 = 2 * tid, i1 = 2 * tid + 1;
  } else {
    i0 = tid, i1 = tid + hs / 2;
  }
  AttnIn in{0.f, 0.f, 0.f, 0.f, 0.f};
  if (handoff) {
    const unsigned long long* pv = ph.tv + kvh * hs + tid;
    const unsigned long long* pq0 = ph.tq + head * hs + i0;
    const unsigned long long* pq1 = ph.tq + head * hs + i1;
    const unsigned long long* any = need_q ? pq0 : pv;  // a word this thread waits for anyway
    in = poll_attention_inputs(need_q ? pq0 : any, need_q ? pq1 : any, need_k ? ph.tk + kvh * hs + i0 : any,
                               need_k ? ph.tk + kvh * hs + i1 : any, need_v ? pv : any, tag_in);
  } else {
    if (need_q) in.q0 = __ldcg(P.q + static_cast<size_t>(head) * hs + i0), in.q1 = __ldcg(P.q + static_cast<size_t>(head) * hs + i1);
    if (need_k) in.k0 = __ldcg(P.k_raw + kvh * hs + i0), in.k1 = __ldcg(P.k_raw + kvh * hs + i1);
    if (need_v) in.v = __ldcg(v_plain);
  }
  if (need_q) {
    const int ci = 2 * tid;
    const float fci = P.sin_cache[static_cast<size_t>(pos) * hs + ci];
    const float fcr = P.cos_cache[static_cast<size_t>(pos) * hs + ci];
    q_s[i0] = __fmaf_rn(fcr, in.q0, -__fmul_rn(fci, in.q1));
    q_s[i1] = __fmaf_rn(fci, in.q0, __fmul_rn(fcr, in.q1));
    if (need_k) {
      const float r0 = __fmaf_rn(fcr, in.k0, -__fmul_rn(fci, in.k1));
      const float r1 = __fmaf_rn(fci, in.k0, __fmul_rn(fcr, in.k1));
      k_s[i0] = r0;
      k_s[i1] = r1;
      if (head % P.kv_mul == 0) {  // one writer per kv head stores the rotated key
        kcache[(static_cast<size_t>(i0 >> 2) * seq_len + pos) * 4 + (i0 & 3)] = r0;
        kcache[(static_cast<size_t>(i1 >> 2) * seq_len + pos) * 4 + (i1 & 3)] = r1;
      }
    }
  }
  return need_v ? in.v : 0.f;
}

// ---- attention: SP CTAs per query head, two phases (mha_kernel.cu:47-110 + rope_kernel.cu) ---------
// The reference gives a head one CTA and so did round 1: 32 of 148 SMs worked while the rest polled,
// and the time grew with the context.  Every score (one left-to-right FFMA chain per timestep) and
// every output element (one FFMA chain over the timesteps) is independent of the others, so the work
// splits over SP CTAs per head WITHOUT touching a single chain -- results stay bit-identical:
//   scores phase  CTA (head, s) rotates q (and the new key row), takes the K tiles j = s, s + SP, ...
//                 and publishes its scaled scores as tagged words scores[head][t];
//   P.V phase     CTA (head, s) polls all pos + 1 scores of the head, runs the softmax (every CTA of
//                 the head the same bits), and owns output dims [s dv, (s + 1) dv), dv = head_size / SP:
//                 it streams only that slice of V and publishes its dv outputs.
// KV layout (persistent engine only; kllm_decoder_read_kv converts back):
//   K [L][kv_head][head_size/4][seq_len][4]   -- 16-byte chunk c of timestep t at ((c*seq_len)+t)*4:
//       a tile of T timesteps is hs/4 contiguous runs of T*16 bytes, and "thread t reads chunk c"
//       is a conflict-free 128-bit shared-memory access (consecutive t -> consecutive 16 B);
//   V [L][kv_head][SP][seq_len][dv]           -- a tile of T timesteps of one slice is one contiguous
//       block and "thread i walks column i" is conflict-free.
// Rows t < pos were written by earlier tokens, so -- like weights -- the producer warp streams
// them through the ring ahead of time; only row pos is handled here from registers.
constexpr bool kAttnGate = KLLM_ATTN_GATE != 0;
__device__ __forceinline__ int attn_tiles(int pos, int T) { return (pos + T - 1) / T; }
// tiles j = s, s + SP, ... < n
__device__ __forceinline__ int own_tiles(int n, int s, int SP) { return n > s ? (n - s + SP - 1) / SP : 0; }

// One output element's P.V chain over nt timesteps of a staged tile: value += pr[tt] * vt[tt * stride],
// strictly left to right (mha_kernel.cu:97-109).  The chain is latency bound (one dependent FFMA per
// step), so the operands of the next eight steps are loaded while the current eight retire.
// pv_chain_smem: probabilities in shared memory (the usual case) -- explicit ld.shared, the eight
// probabilities of a batch as two 128-bit loads (pr_addr is 16-byte aligned: tiles start at
// multiples of 32 timesteps).  pv_chain: probabilities behind a generic pointer (global fallback).
__device__ __forceinline__ float pv_chain_smem(uint32_t pr_addr, uint32_t vt_addr, int stride_bytes, int nt, float value) {
  // two register sets (A: steps tt .. tt+7, B: tt+8 .. tt+15) loaded alternately, so the loop carries no
  // register moves and every load has a whole 8-step chain (>= 32 cycles) to land
  auto load8 = [&](int t, float4& p0, float4& p1, float (&v)[8]) {
    p0 = lds_f4(pr_addr + t * 4), p1 = lds_f4(pr_addr + t * 4 + 16);
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = lds_f32(vt_addr + (t + k) * stride_bytes);
  };
  auto chain8 = [&](const float4& p0, const float4& p1, const float (&v)[8]) {
    value = __fmaf_rn(p0.x, v[0], value);
    value = __fmaf_rn(p0.y, v[1], value);
    value = __fmaf_rn(p0.z, v[2], value);
    value = __fmaf_rn(p0.w, v[3], value);
    value = __fmaf_rn(p1.x, v[4], value);
    value = __fmaf_rn(p1.y, v[5], value);
    value = __fmaf_rn(p1.z, v[6], value);
    value = __fmaf_rn(p1.w, v[7], value);
  };
  int tt = 0;
  if (nt >= 8) {
    float4 a0, a1, b0, b1;
    float va[8], vb[8];
    load8(0, a0, a1, va);
    for (; tt + 24 <= nt; tt += 16) {  // A holds tt .. tt+7
      load8(tt + 8, b0, b1, vb);
      chain8(a0, a1, va);
      load8(tt + 16, a0, a1, va);
      chain8(b0, b1, vb);
    }
    if (tt + 16 <= nt) {
      load8(tt + 8, b0, b1, vb);
      chain8(a0, a1, va);
      chain8(b0, b1, vb);
      tt += 16;
    } else {
      chain8(a0, a1, va);
      tt += 8;
    }
  }
  for (; tt < nt; ++tt) value = __fmaf_rn(lds_f32(pr_addr + tt * 4), lds_f32(vt_addr + tt * stride_bytes), value);
  return value;
}
__device__ __forceinline__ float pv_chain(const float* pr, const float* vt, int stride, int nt, float value) {
#pragma unroll 8
  for (int tt = 0; tt < nt; ++tt) value = __fmaf_rn(pr[tt], vt[tt * stride], value);
  return value;
}

// Fused form (attn_split == 1, one CTA per head does scores, softmax and P.V in ONE phase): one
// hand-off less per layer, the better trade when a head's K and V are small (head_size 64).
template <int CW>
__device__ KLLM_PHASE_CALL Pipe attention_fused_phase(const Params& P, int head, int pos, Pipe pipe, unsigned tag_in,
                                                 unsigned tag_out, unsigned long long* stamp) {
  const Phase& ph = g_ph_cons;
  float* ws = reinterpret_cast<float*>(smem);
  float* s_warp = g_s_warp;
  float* s_bcast = &g_s_bcast;
  unsigned char* stages = smem + P.xbuf_bytes + P.xres_bytes;
  uint64_t* full_bar = g_full_bar;
  uint64_t* empty_bar = g_empty_bar;
  constexpr int CT = CW * 32;
  const int tid = threadIdx.x;
  const long long c_begin = stamp ? clock64() : 0;
  long long c_wait = 0;
  const int lane = tid & 31, warp = tid >> 5;
  const int hs = P.head_size, seq_len = P.seq_len, T = P.attn_tile, S = P.num_stages;
  float* q_s = ws;       // [hs] rotated query
  float* k_s = ws + hs;  // [hs] rotated key of the current position
  const int kvh = head / P.kv_mul;
  const size_t head_block = (static_cast<size_t>(ph.layer) * (P.kv_dim / hs) + kvh) * seq_len * hs;
  float* kcache = P.key_cache + head_block;
  const float* vcache = P.value_cache + head_block;
  // scores / probabilities: shared memory when the context fits the workspace (the ring leaves
  // almost no L1), else the global [head][seq_len] buffer the reference uses
  const int smem_cap = (P.xbuf_bytes >> 2) - 2 * hs;
  const bool score_in_smem = pos + 1 <= smem_cap;
  float* score_head = score_in_smem ? (ws + 2 * hs) : (P.score + static_cast<size_t>(head) * seq_len);

  // q, the new key row (rotated) and the value row of the current position (QKV phase of this token)
  const float v_pos = attention_inputs(P, ph, head, kvh, pos, tag_in, true, true, q_s, k_s, kcache,
                                       vcache + static_cast<size_t>(pos) * hs + tid);
  consumer_sync<CT>();
  const long long c_rope = stamp ? clock64() : 0;

  // ---- scores: one left-to-right FFMA chain per timestep (mha_kernel.cu:61-91) ---------------
  const float scale = 1.f / sqrtf(static_cast<float>(hs));
  const float4* q4 = reinterpret_cast<const float4*>(q_s);
  const int n_tiles = attn_tiles(pos, T);
  for (int j = 0; j < n_tiles; ++j) {
    const int t0 = j * T;
    const int nt = min(T, pos - t0);
    // warps without a row in this tile do not wait for it (a spinning warp costs its neighbours
    // issue slots and shared-memory queue entries): they arrive at once and block at the hardware
    // barrier below, which also keeps them from lapping the ring
    const bool works = !kAttnGate || ((tid & ~31) < nt);
    if (works) {
      const long long w0 = stamp ? clock64() : 0;
      mbar_wait(&full_bar[pipe.slot], pipe.parity);
      if (stamp) c_wait += clock64() - w0;
    }
    const float4* tile = reinterpret_cast<const float4*>(stages + static_cast<size_t>(pipe.slot) * P.stage_bytes);
    if (tid < nt) {
      float score = 0.0f;
#pragma unroll 4
      for (int c = 0; c < (hs >> 2); ++c) {
        const float4 kv = tile[c * T + tid];
        const float4 qv = q4[c];
        score = __fmaf_rn(kv.x, qv.x, score);
        score = __fmaf_rn(kv.y, qv.y, score);
        score = __fmaf_rn(kv.z, qv.z, score);
        score = __fmaf_rn(kv.w, qv.w, score);
      }
      score_head[t0 + tid] = __fmul_rn(score, scale);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty_bar[pipe.slot]);
    pipe.advance(S);
    if (kAttnGate) consumer_sync<CT>();
  }
  if (tid == 0) {  // t == pos from the freshly rotated key
    const float4* k4 = reinterpret_cast<const float4*>(k_s);
    float score = 0.0f;
    for (int c = 0; c < (hs >> 2); ++c) {
      const float4 kv = k4[c];
      const float4 qv = q4[c];
      score = __fmaf_rn(kv.x, qv.x, score);
      score = __fmaf_rn(kv.y, qv.y, score);
      score = __fmaf_rn(kv.z, qv.z, score);
      score = __fmaf_rn(kv.w, qv.w, score);
    }
    score_head[pos] = __fmul_rn(score, scale);
  }
  consumer_sync<CT>();
  const long long c_scores = stamp ? clock64() : 0;
  const long long c_wait_scores = c_wait;

  // ---- softmax, mha_kernel.cu:7-45: the reference runs 256 strided threads and cub<256> block
  // reductions.  Here 128 threads play two virtual threads each (v = tid and v = tid + 128, i.e.
  // elements tid + 256 k and tid + 128 + 256 k): the maximum does not care about order, and for the
  // sum each virtual thread keeps its own left-to-right partial, each virtual warp its own shuffle
  // tree (real warp q holds virtual warps q and q + 4), then the eight warp sums are added in order.
  const int size = pos + 1;
  constexpr int kHalf = kSoftmaxThreads / 2;  // 128 real threads
  static_assert(CT >= kHalf, "softmax needs 128 consumer threads");
  const bool sm_thread = tid < kHalf;
  float max_val = -FLT_MAX;
  if (sm_thread)
    for (int i = tid; i < size; i += kHalf) max_val = fmaxf(max_val, score_head[i]);
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) max_val = fmaxf(max_val, __shfl_xor_sync(kFull, max_val, off));
  if (lane == 0 && sm_thread) s_warp[warp] = max_val;
  consumer_sync<CT>();
  max_val = fmaxf(fmaxf(s_warp[0], s_warp[1]), fmaxf(s_warp[2], s_warp[3]));
  consumer_sync<CT>();

  float sum_lo = 0.0f, sum_hi = 0.0f;  // virtual threads tid and tid + 128
  if (sm_thread) {
    for (int i = tid; i < size; i += kSoftmaxThreads) {
      const float e = expf(score_head[i] - max_val);
      score_head[i] = e;
      sum_lo += e;
    }
    for (int i = tid + kHalf; i < size; i += kSoftmaxThreads) {
      const float e = expf(score_head[i] - max_val);
      score_head[i] = e;
      sum_hi += e;
    }
  }
  sum_lo = warp_tree_sum(sum_lo);
  sum_hi = warp_tree_sum(sum_hi);
  if (lane == 0 && sm_thread) {
    s_warp[warp] = sum_lo;      // virtual warp `warp`
    s_warp[warp + 4] = sum_hi;  // virtual warp `warp + 4`
  }
  consumer_sync<CT>();
  if (tid == 0) {
    float total = s_warp[0];
#pragma unroll
    for (int w = 1; w < kSoftmaxThreads / 32; ++w) total = __fadd_rn(total, s_warp[w]);
    *s_bcast = total;
  }
  consumer_sync<CT>();
  const float sum = *s_bcast;
  for (int i = tid; i < size; i += CT) score_head[i] = score_head[i] / sum;
  consumer_sync<CT>();
  const long long c_soft = stamp ? clock64() : 0;

  // ---- weighted value sum, mha_kernel.cu:97-109: one FFMA chain per output element ----------------
  float value = 0.0f;
  const int Tv = P.attn_tile_v, n_tiles_v = attn_tiles(pos, Tv);
  for (int j = 0; j < n_tiles_v; ++j) {
    const int t0 = j * Tv;
    const int nt = min(Tv, pos - t0);
    // warps without a row in this tile do not wait for it (a spinning warp costs its neighbours
    // issue slots and shared-memory queue entries): they arrive at once and block at the hardware
    // barrier below, which also keeps them from lapping the ring
    const bool works = !kAttnGate || ((tid & ~31) < hs);
    if (works) {
      const long long w0 = stamp ? clock64() : 0;
      mbar_wait(&full_bar[pipe.slot], pipe.parity);
      if (stamp) c_wait += clock64() - w0;
    }
    if (tid < hs) {
      const float* vt = reinterpret_cast<const float*>(stages + static_cast<size_t>(pipe.slot) * P.stage_bytes) + tid;
      value = score_in_smem ? pv_chain_smem(smem_u32(score_head + t0), smem_u32(vt), hs * 4, nt, value)
                            : pv_chain(score_head + t0, vt, hs, nt, value);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty_bar[pipe.slot]);
    pipe.advance(S);
    if (kAttnGate) consumer_sync<CT>();
  }
  if (tid < hs) {
    value = __fmaf_rn(score_head[pos], v_pos, value);
    if (ph.ta != nullptr)
      st_tagged_gpu(ph.ta + static_cast<size_t>(head) * hs + tid, value, tag_out);
    else
      P.attn_out[static_cast<size_t>(head) * hs + tid] = value;
  }
  if (stamp && tid == 0) {  // SM cycles of thread 0 (profiles/: tools/phase_timeline.py)
    const long long c_end = clock64();
    stamp[4] = static_cast<unsigned long long>(c_rope - c_begin);                             // q/k/v poll + RoPE
    stamp[5] = static_cast<unsigned long long>(c_scores - c_rope - c_wait_scores);            // scores
    stamp[6] = static_cast<unsigned long long>(c_soft - c_scores);                            // softmax
    stamp[7] = static_cast<unsigned long long>(c_end - c_soft - (c_wait - c_wait_scores));    // P.V
    stamp[8] = static_cast<unsigned long long>(c_wait);                                       // ring waits
    stamp[9] = static_cast<unsigned long long>(c_wait - c_wait_scores);                       // of which V tiles
  }
  return pipe;
}


template <int CW>
__device__ KLLM_PHASE_CALL Pipe attention_scores_phase(const Params& P, int head, int split, int pos, Pipe pipe,
                                                        unsigned tag_in, unsigned tag_out, unsigned long long* stamp) {
  const Phase& ph = g_ph_cons;
  float* ws = reinterpret_cast<float*>(smem);
  unsigned char* stages = smem + P.xbuf_bytes + P.xres_bytes;
  uint64_t* full_bar = g_full_bar;
  uint64_t* empty_bar = g_empty_bar;
  constexpr int CT = CW * 32;
  const int tid = threadIdx.x;
  const long long c_begin = stamp ? clock64() : 0;
  long long c_wait = 0;
  const int lane = tid & 31;
  const int hs = P.head_size, seq_len = P.seq_len, T = P.attn_tile, S = P.num_stages, SP = P.attn_split;
  float* q_s = ws;       // [hs] rotated query
  float* k_s = ws + hs;  // [hs] rotated key of the current position
  const int kvh = head / P.kv_mul;
  const size_t head_block = (static_cast<size_t>(ph.layer) * (P.kv_dim / hs) + kvh) * seq_len * hs;
  float* kcache = P.key_cache + head_block;
  unsigned long long* sc_out = P.scores + static_cast<size_t>(head) * seq_len;
  // q and -- in the CTA that scores it -- the new key row, rotated (the value row is the P.V phase's business)
  attention_inputs(P, ph, head, kvh, pos, tag_in, split == 0, false, q_s, k_s, kcache, nullptr);
  consumer_sync<CT>();
  const long long c_rope = stamp ? clock64() : 0;

  // ---- scores: one left-to-right FFMA chain per timestep (mha_kernel.cu:61-91) ---------------
  const float scale = 1.f / sqrtf(static_cast<float>(hs));
  const float4* q4 = reinterpret_cast<const float4*>(q_s);
  const int n_tiles = attn_tiles(pos, T);
  for (int j = split; j < n_tiles; j += SP) {
    const int t0 = j * T;
    const int nt = min(T, pos - t0);
    // warps without a row in this tile do not wait for it (a spinning warp costs its neighbours
    // issue slots and shared-memory queue entries): they arrive at once and block at the hardware
    // barrier below, which also keeps them from lapping the ring
    const bool works = !kAttnGate || ((tid & ~31) < nt);
    if (works) {
      const long long w0 = stamp ? clock64() : 0;
      mbar_wait(&full_bar[pipe.slot], pipe.parity);
      if (stamp) c_wait += clock64() - w0;
    }
    const float4* tile = reinterpret_cast<const float4*>(stages + static_cast<size_t>(pipe.slot) * P.stage_bytes);
    if (tid < nt) {
      float score = 0.0f;
#pragma unroll 4
      for (int c = 0; c < (hs >> 2); ++c) {
        const float4 kv = tile[c * T + tid];
        const float4 qv = q4[c];
        score = __fmaf_rn(kv.x, qv.x, score);
        score = __fmaf_rn(kv.y, qv.y, score);
        score = __fmaf_rn(kv.z, qv.z, score);
        score = __fmaf_rn(kv.w, qv.w, score);
      }
      st_tagged_gpu(sc_out + t0 + tid, __fmul_rn(score, scale), tag_out);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty_bar[pipe.slot]);
    pipe.advance(S);
    if (kAttnGate) consumer_sync<CT>();
  }
  if (split == 0 && tid == 0) {  // t == pos from the freshly rotated key
    const float4* k4 = reinterpret_cast<const float4*>(k_s);
    float score = 0.0f;
    for (int c = 0; c < (hs >> 2); ++c) {
      const float4 kv = k4[c];
      const float4 qv = q4[c];
      score = __fmaf_rn(kv.x, qv.x, score);
      score = __fmaf_rn(kv.y, qv.y, score);
      score = __fmaf_rn(kv.z, qv.z, score);
      score = __fmaf_rn(kv.w, qv.w, score);
    }
    st_tagged_gpu(sc_out + pos, __fmul_rn(score, scale), tag_out);
  }
  if (stamp && tid == 0) {
    const long long c_end = clock64();
    stamp[4] = static_cast<unsigned long long>(c_rope - c_begin);           // q/k poll + RoPE
    stamp[5] = static_cast<unsigned long long>(c_end - c_rope - c_wait);    // scores
    stamp[8] = static_cast<unsigned long long>(c_wait);                     // ring waits (K tiles)
  }
  return pipe;
}

template <int CW>
__device__ KLLM_PHASE_CALL Pipe attention_pv_phase(const Params& P, int head, int split, int pos, Pipe pipe,
                                                   unsigned tag_scores, unsigned tag_qkv, unsigned tag_out,
                                                   unsigned long long* stamp) {
  const Phase& ph = g_ph_cons;
  float* ws = reinterpret_cast<float*>(smem);
  float* s_warp = g_s_warp;
  float* s_bcast = &g_s_bcast;
  unsigned char* stages = smem + P.xbuf_bytes + P.xres_bytes;
  uint64_t* full_bar = g_full_bar;
  uint64_t* empty_bar = g_empty_bar;
  constexpr int CT = CW * 32;
  const int tid = threadIdx.x;
  const long long c_begin = stamp ? clock64() : 0;
  long long c_wait = 0;
  const int lane = tid & 31, warp = tid >> 5;
  const int hs = P.head_size, seq_len = P.seq_len, S = P.num_stages, SP = P.attn_split;
  const int dv = hs / SP, T = P.attn_tile_v;
  const int kvh = head / P.kv_mul;
  const size_t slice_block =
      ((static_cast<size_t>(ph.layer) * (P.kv_dim / hs) + kvh) * SP + split) * seq_len * dv;
  const float* vslice = P.value_cache + slice_block;
  const bool handoff = ph.tv != nullptr;
  // scores / probabilities: shared memory when the context fits the workspace (the ring leaves
  // almost no L1), else the global [head][seq_len] buffer the reference uses (the SP CTAs of a head
  // then write identical values to it)
  const int smem_cap = P.xbuf_bytes >> 2;
  const bool score_in_smem = pos + 1 <= smem_cap;
  float* score_head = score_in_smem ? ws : (P.score + static_cast<size_t>(head) * seq_len);

  // this CTA's dv dims of the value row of the current position (written by the QKV phase of this token)
  float v_pos = 0.f;
  if (tid < dv)
    v_pos = handoff ? poll_tagged(ph.tv + kvh * hs + split * dv + tid, tag_qkv)
                    : __ldcg(vslice + static_cast<size_t>(pos) * dv + tid);

  // all pos + 1 scaled scores of the head, polled in place
  const int size = pos + 1;
  {
    const unsigned long long* sc_in = P.scores + static_cast<size_t>(head) * seq_len;
    const int n4 = size >> 2;  // seq_len % 4 == 0: the head's words start 32-byte aligned
    stage_handoff<4>(sc_in, tag_scores, n4, tid, CT, reinterpret_cast<float4*>(score_head));
    const int rest = 4 * n4 + tid;
    if (tid < 4 && rest < size) score_head[rest] = poll_tagged(sc_in + rest, tag_scores);
  }
  consumer_sync<CT>();
  const long long c_poll = stamp ? clock64() : 0;

  // ---- softmax, mha_kernel.cu:7-45: the reference runs 256 strided threads and cub<256> block
  // reductions.  Here 128 threads play two virtual threads each (v = tid and v = tid + 128, i.e.
  // elements tid + 256 k and tid + 128 + 256 k): the maximum does not care about order, and for the
  // sum each virtual thread keeps its own left-to-right partial, each virtual warp its own shuffle
  // tree (real warp q holds virtual warps q and q + 4), then the eight warp sums are added in order.
  constexpr int kHalf = kSoftmaxThreads / 2;  // 128 real threads
  static_assert(CT >= kHalf, "softmax needs 128 consumer threads");
  const bool sm_thread = tid < kHalf;
  float max_val = -FLT_MAX;
  if (sm_thread)
    for (int i = tid; i < size; i += kHalf) max_val = fmaxf(max_val, score_head[i]);
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) max_val = fmaxf(max_val, __shfl_xor_sync(kFull, max_val, off));
  if (lane == 0 && sm_thread) s_warp[warp] = max_val;
  consumer_sync<CT>();
  max_val = fmaxf(fmaxf(s_warp[0], s_warp[1]), fmaxf(s_warp[2], s_warp[3]));
  consumer_sync<CT>();

  float sum_lo = 0.0f, sum_hi = 0.0f;  // virtual threads tid and tid + 128
  if (sm_thread) {
    for (int i = tid; i < size; i += kSoftmaxThreads) {
      const float e = expf(score_head[i] - max_val);
      score_head[i] = e;
      sum_lo += e;
    }
    for (int i = tid + kHalf; i < size; i += kSoftmaxThreads) {
      const float e = expf(score_head[i] - max_val);
      score_head[i] = e;
      sum_hi += e;
    }
  }
  sum_lo = warp_tree_sum(sum_lo);
  sum_hi = warp_tree_sum(sum_hi);
  if (lane == 0 && sm_thread) {
    s_warp[warp] = sum_lo;      // virtual warp `warp`
    s_warp[warp + 4] = sum_hi;  // virtual warp `warp + 4`
  }
  consumer_sync<CT>();
  if (tid == 0) {
    float total = s_warp[0];
#pragma unroll
    for (int w = 1; w < kSoftmaxThreads / 32; ++w) total = __fadd_rn(total, s_warp[w]);
    *s_bcast = total;
  }
  consumer_sync<CT>();
  const float sum = *s_bcast;
  for (int i = tid; i < size; i += CT) score_head[i] = score_head[i] / sum;
  consumer_sync<CT>();
  const long long c_soft = stamp ? clock64() : 0;

  // ---- weighted value sum, mha_kernel.cu:97-109: one FFMA chain per output element ----------------
  float value = 0.0f;
  const int n_tiles = attn_tiles(pos, T);
  for (int j = 0; j < n_tiles; ++j) {
    const int t0 = j * T;
    const int nt = min(T, pos - t0);
    // warps without a row in this tile do not wait for it (a spinning warp costs its neighbours
    // issue slots and shared-memory queue entries): they arrive at once and block at the hardware
    // barrier below, which also keeps them from lapping the ring
    const bool works = !kAttnGate || ((tid & ~31) < dv);
    if (works) {
      const long long w0 = stamp ? clock64() : 0;
      mbar_wait(&full_bar[pipe.slot], pipe.parity);
      if (stamp) c_wait += clock64() - w0;
    }
    if (tid < dv) {
      const float* vt = reinterpret_cast<const float*>(stages + static_cast<size_t>(pipe.slot) * P.stage_bytes) + tid;
      value = score_in_smem ? pv_chain_smem(smem_u32(score_head + t0), smem_u32(vt), dv * 4, nt, value)
                            : pv_chain(score_head + t0, vt, dv, nt, value);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty_bar[pipe.slot]);
    pipe.advance(S);
    if (kAttnGate) consumer_sync<CT>();
  }
  if (tid < dv) {
    value = __fmaf_rn(score_head[pos], v_pos, value);
    const int d = split * dv + tid;
    if (ph.ta != nullptr)
      st_tagged_gpu(ph.ta + static_cast<size_t>(head) * hs + d, value, tag_out);
    else
      P.attn_out[static_cast<size_t>(head) * hs + d] = value;
  }
  if (stamp && tid == 0) {
    const long long c_end = clock64();
    stamp[4] = static_cast<unsigned long long>(c_poll - c_begin);           // scores (+ v row) polled
    stamp[6] = static_cast<unsigned long long>(c_soft - c_poll);            // softmax
    stamp[7] = static_cast<unsigned long long>(c_end - c_soft - c_wait);    // P.V
    stamp[8] = static_cast<unsigned long long>(c_wait);                     // ring waits (V tiles)
  }
  return pipe;
}

// Toleranced attention (numerics "fast"): flash-decoding.  With the summation order free, a head is
// split over SP CTAs BY TIMESTEP -- CTA (head, s) takes the tiles j = s, s + SP, ... of T timesteps, K
// and V -- and inside the CTA every WARP runs its own online softmax over blocks of 8 timesteps
// (blocks dealt round-robin to the warps), so a tile costs no block-wide barrier at all:
//   scores   lane (cg, tt) = (lane / 8, lane % 8) dots timestep tt of the block with a quarter of
//            head_size (conflict-free 128-bit reads of the K tile [hs/4][T][4]); two xor-shuffles sum
//            the quarters, three more give the block's maximum and sum -> running (m, l) of the warp;
//   P.V      lane owns output dims lane, lane + 32, ...: o[d] = o[d] alpha + sum_tt p_tt v[tt][d] with p_tt
//            shuffled from lane tt (conflict-free 32-bit reads of the V tile [T][hs]).
// At the end the CW warp partials (m, l, o[hs]) are merged through shared memory, CTA 0 of the head folds
// in the current position's row from registers and merges the partials of the other CTAs that had
// tiles (tagged words in the scores area: [head][s][hs + 2]); at short contexts (pos <= T) that is
// nobody, and the phase costs what the fused one does.
template <int CW>
__device__ KLLM_PHASE_CALL Pipe attention_flash_phase(const Params& P, int head, int split, int pos, Pipe pipe,
                                                       unsigned tag_in, unsigned tag_out, unsigned long long* stamp) {
  const Phase& ph = g_ph_cons;
  float* ws = reinterpret_cast<float*>(smem);
  unsigned char* stages = smem + P.xbuf_bytes + P.xres_bytes;
  uint64_t* full_bar = g_full_bar;
  uint64_t* empty_bar = g_empty_bar;
  constexpr int CT = CW * 32;
  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  const long long c_begin = stamp ? clock64() : 0;
  long long c_wait = 0, c_sc = 0, c_pv = 0;
  const int hs = P.head_size, seq_len = P.seq_len, T = P.attn_tile, S = P.num_stages, SP = P.attn_split;
  const int n_tiles = attn_tiles(pos, T);
  // CTAs without a tile have nothing to say (their partial would weigh zero): only CTA 0 always runs
  if (split != 0 && split >= n_tiles) return pipe;
  float* q_s = ws;                // [hs] rotated query
  float* k_s = ws + hs;           // [hs] rotated key of the current position
  float* red = ws + 2 * hs;       // [CW][hs + 2] warp partials: m, l, o[hs]
  const int kvh = head / P.kv_mul;
  const size_t head_block = (static_cast<size_t>(ph.layer) * (P.kv_dim / hs) + kvh) * seq_len * hs;
  float* kcache = P.key_cache + head_block;
  // q, and in CTA 0 of the head the new key row (rotated) and the value row of the current position
  const float v_pos = attention_inputs(P, ph, head, kvh, pos, tag_in, split == 0, split == 0, q_s, k_s, kcache,
                                       P.value_cache + head_block + static_cast<size_t>(pos) * hs + tid);
  consumer_sync<CT>();
  const long long c_rope = stamp ? clock64() : 0;

  const float scale = 1.f / sqrtf(static_cast<float>(hs));
  const float4* q4 = reinterpret_cast<const float4*>(q_s);
  const int cg = lane >> 3, tt = lane & 7;
  const int cpg = hs >> 4;        // 16-byte chunks per quarter of head_size (host: head_size % 16 == 0)
  float m = -FLT_MAX, l = 0.f;
  float o[4] = {0.f, 0.f, 0.f, 0.f};  // output dims lane, lane + 32, lane + 64, lane + 96 (< hs)
  int blk0 = 0;                   // blocks dealt so far: block b of the CTA goes to warp b % CW
  for (int j = split; j < n_tiles; j += SP) {
    const int t0 = j * T;
    const int nt = min(T, pos - t0);
    const long long w0 = stamp ? clock64() : 0;
    mbar_wait(&full_bar[pipe.slot], pipe.parity);  // K tile
    const uint32_t ktile = smem_u32(stages + static_cast<size_t>(pipe.slot) * P.stage_bytes);
    const int kslot = pipe.slot;
    pipe.advance(S);
    mbar_wait(&full_bar[pipe.slot], pipe.parity);  // V tile
    const uint32_t vtile = smem_u32(stages + static_cast<size_t>(pipe.slot) * P.stage_bytes);
    const long long w1 = stamp ? clock64() : 0;
    c_wait += w1 - w0;
    const int nb = (nt + 7) >> 3;
    for (int b = (warp - blk0 % CW + CW) % CW; b < nb; b += CW) {
      const long long s0 = stamp ? clock64() : 0;
      const int tl = b * 8 + tt;  // this lane's timestep within the tile
      const bool valid = tl < nt;
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
      if (valid) {
#pragma unroll 4
        for (int c = cg * cpg; c < (cg + 1) * cpg; ++c) {
          const float4 kv = lds_f4(ktile + static_cast<uint32_t>(c * T + tl) * 16u);
          const float4 qv = q4[c];
          a0 = __fmaf_rn(kv.x, qv.x, a0);
          a1 = __fmaf_rn(kv.y, qv.y, a1);
          a2 = __fmaf_rn(kv.z, qv.z, a2);
          a3 = __fmaf_rn(kv.w, qv.w, a3);
        }
      }
      float sc = (a0 + a1) + (a2 + a3);
      sc += __shfl_xor_sync(kFull, sc, 8);
      sc += __shfl_xor_sync(kFull, sc, 16);
      sc = valid ? sc * scale : -FLT_MAX;
      float mb = sc;
      mb = fmaxf(mb, __shfl_xor_sync(kFull, mb, 1));
      mb = fmaxf(mb, __shfl_xor_sync(kFull, mb, 2));
      mb = fmaxf(mb, __shfl_xor_sync(kFull, mb, 4));
      const float m_new = fmaxf(m, mb);
      const float alpha = expf(m - m_new);
      const float pr = valid ? expf(sc - m_new) : 0.f;
      float ps = pr;
      ps += __shfl_xor_sync(kFull, ps, 1);
      ps += __shfl_xor_sync(kFull, ps, 2);
      ps += __shfl_xor_sync(kFull, ps, 4);
      l = __fmaf_rn(l, alpha, ps);
      m = m_new;
      const long long s1 = stamp ? clock64() : 0;
      c_sc += s1 - s0;
      // P.V of the block
      const int nv = min(8, nt - b * 8);
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
      const uint32_t vrow = vtile + static_cast<uint32_t>(b * 8 * hs + lane) * 4u;
      for (int k = 0; k < nv; ++k) {
        const float pk = __shfl_sync(kFull, pr, k);
        const uint32_t va = vrow + static_cast<uint32_t>(k * hs) * 4u;
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (lane + 32 * i < hs) acc[i] = __fmaf_rn(pk, lds_f32(va + 128u * i), acc[i]);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) o[i] = __fmaf_rn(o[i], alpha, acc[i]);
      if (stamp) c_pv += clock64() - s1;
    }
    blk0 += nb;
    __syncwarp();
    if (lane == 0) {
      mbar_arrive(&empty_bar[kslot]);
      mbar_arrive(&empty_bar[pipe.slot]);
    }
    pipe.advance(S);
  }
  const long long c_tiles = stamp ? clock64() : 0;
  // ---- merge the warps' partials: thread d < hs ends with the CTA's (m, l, o[d]) ---------------------
  {
    float* mine = red + warp * (hs + 2);
    if (lane == 0) mine[0] = m, mine[1] = l;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (lane + 32 * i < hs) mine[2 + lane + 32 * i] = o[i];
  }
  consumer_sync<CT>();
  if (tid < hs) {
    float M = red[0];
    for (int w = 1; w < CW; ++w) M = fmaxf(M, red[w * (hs + 2)]);
    float num = 0.f, den = 0.f;
    for (int w = 0; w < CW; ++w) {
      const float* theirs = red + w * (hs + 2);
      const float wgt = expf(theirs[0] - M);
      num = __fmaf_rn(theirs[2 + tid], wgt, num);
      den = __fmaf_rn(theirs[1], wgt, den);
    }
    if (split == 0) {  // the current position, from the freshly rotated key and the polled value row
      const float4* k4 = reinterpret_cast<const float4*>(k_s);
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
      for (int c = 0; c < (hs >> 2); ++c) {
        const float4 kv = k4[c];
        const float4 qv = q4[c];
        a0 = __fmaf_rn(kv.x, qv.x, a0);
        a1 = __fmaf_rn(kv.y, qv.y, a1);
        a2 = __fmaf_rn(kv.z, qv.z, a2);
        a3 = __fmaf_rn(kv.w, qv.w, a3);
      }
      const float s_pos = ((a0 + a1) + (a2 + a3)) * scale;
      const float M_new = fmaxf(M, s_pos);
      const float alpha = expf(M - M_new);
      const float pp = expf(s_pos - M_new);
      num = __fmaf_rn(num, alpha, pp * v_pos);
      den = __fmaf_rn(den, alpha, pp);
      M = M_new;
    }
    unsigned long long* area = P.scores + static_cast<size_t>(head) * seq_len;  // [SP][hs + 2] tagged words
    if (split != 0) {
      unsigned long long* mine = area + static_cast<size_t>(split) * (hs + 2);
      st_tagged_gpu(mine + 2 + tid, num, tag_out);
      if (tid == 0) st_tagged2_gpu(mine, M, den, tag_out);
    } else {
      const int active = min(SP, n_tiles);  // CTAs 1 .. active - 1 of the head had tiles
      // their partials, up to three CTAs' (m, l, o[tid]) in flight together: polled one CTA after the other
      // every partial would be another L2 round trip on the layer's critical path
      for (int s0 = 1; s0 < active; s0 += 3) {
        unsigned long long w_m[3], w_l[3], w_o[3];
        const int ns = min(3, active - s0);
        const long long t_start = clock64();
        for (;;) {
          bool ok = true;
          unsigned seen = tag_out;
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            const unsigned long long* theirs = area + static_cast<size_t>(s0 + min(k, ns - 1)) * (hs + 2);
            ld_tagged2_gpu(theirs, w_m[k], w_l[k]);
            w_o[k] = ld_tagged_gpu(theirs + 2 + tid);
          }
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            if (tag_of(w_m[k]) != tag_out) ok = false, seen = tag_of(w_m[k]);
            if (tag_of(w_l[k]) != tag_out) ok = false, seen = tag_of(w_l[k]);
            if (tag_of(w_o[k]) != tag_out) ok = false, seen = tag_of(w_o[k]);
          }
          if (ok) break;
          poll_failed(seen, tag_out, t_start, 0);
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          if (k < ns) {  // in CTA order, as before
            const float ms = val_of(w_m[k]), ls = val_of(w_l[k]), os = val_of(w_o[k]);
            const float M_new = fmaxf(M, ms);
            const float fa = expf(M - M_new), fb = expf(ms - M_new);
            num = __fmaf_rn(num, fa, os * fb);
            den = __fmaf_rn(den, fa, ls * fb);
            M = M_new;
          }
        }
      }
      const float value = num / den;
      if (ph.ta != nullptr)
        st_tagged_gpu(ph.ta + static_cast<size_t>(head) * hs + tid, value, tag_out);
      else
        P.attn_out[static_cast<size_t>(head) * hs + tid] = value;
    }
  }
  if (stamp && tid == 0) {
    const long long c_end = clock64();
    stamp[4] = static_cast<unsigned long long>(c_rope - c_begin);  // q/k/v poll + RoPE
    stamp[5] = static_cast<unsigned long long>(c_sc);              // scores + online softmax (warp 0's blocks)
    stamp[6] = static_cast<unsigned long long>(c_end - c_tiles);   // merges: warps, current row, other CTAs
    stamp[7] = static_cast<unsigned long long>(c_pv);              // P.V (warp 0's blocks)
    stamp[8] = static_cast<unsigned long long>(c_wait);            // ring waits
  }
  return pipe;
}

// ---- staging of a tagged input vector ------------------------------------------------------------
// Residual exchange (tp_in): x = x_old + (p_0 + ... + p_{W-1}); the partials of every rank (this
// one included) arrive as tagged words in this rank's exchange area and are polled in place; x_old
// is the CTA's own copy of the residual stream in shared memory (xres), updated here.  Thread t
// handles packs t, t + NT, ...; UP packs x W ranks x 2 loads are in flight per poll round.
// With W == 1 and FOLD the rmsnorm sum of squares is accumulated in the same pass by the
// kNormThreads threads that own the reference's chains (rmsnorm_kernel.cu:19-32).
template <int W, int UP, bool FOLD>
__device__ KLLM_STAGE_CALL float stage_exchange(const unsigned long long* area, int tp_stride, unsigned tag, int n4,
                                                int t, int NT, float4* xs4, float4* xres4) {
  float ssq = 0.f;
  const long long t_start = clock64();
  for (int pb = t; pb < n4; pb += NT * UP) {
    // Every slot of the batch loads SOMETHING (slots past the end re-read the last pack): a buffer
    // with conditionally written elements is kept in local memory by the compiler, and with the ring
    // taking the whole unified L1 a local-memory access is an L2 round trip per poll round.
    unsigned long long wd[UP][W][4];
    bool ok;
    unsigned seen = tag;
    do {
      ok = true;
#pragma unroll
      for (int k = 0; k < UP; ++k) {
        const int p = min(pb + k * NT, n4 - 1);
#pragma unroll
        for (int r = 0; r < W; ++r) {
          const unsigned long long* row = area + static_cast<size_t>(r) * tp_stride + 4 * p;
          if (W == 1) {
            ld_tagged2_gpu(row, wd[k][r][0], wd[k][r][1]);
            ld_tagged2_gpu(row + 2, wd[k][r][2], wd[k][r][3]);
          } else {
            ld_tagged2(row, wd[k][r][0], wd[k][r][1]);
            ld_tagged2(row + 2, wd[k][r][2], wd[k][r][3]);
          }
        }
      }
#pragma unroll
      for (int k = 0; k < UP; ++k)
#pragma unroll
        for (int r = 0; r < W; ++r)
#pragma unroll
          for (int e = 0; e < 4; ++e)
            if (tag_of(wd[k][r][e]) != tag) {
              ok = false;
              seen = tag_of(wd[k][r][e]);
            }
      if (!ok) poll_failed(seen, tag, t_start, 1);
    } while (!ok);
#pragma unroll
    for (int k = 0; k < UP; ++k) {
      const int p = pb + k * NT;
      if (p < n4) {
        float s[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          s[e] = val_of(wd[k][0][e]);
#pragma unroll
          for (int r = 1; r < W; ++r) s[e] = __fadd_rn(s[e], val_of(wd[k][r][e]));  // rank order
        }
        float4 x = xres4[p];
        x.x = __fadd_rn(x.x, s[0]);  // llama3.cpp:683,719: x + out
        x.y = __fadd_rn(x.y, s[1]);
        x.z = __fadd_rn(x.z, s[2]);
        x.w = __fadd_rn(x.w, s[3]);
        xres4[p] = x;
        xs4[p] = x;
        if (FOLD) {
          ssq = __fmaf_rn(x.x, x.x, ssq);
          ssq = __fmaf_rn(x.y, x.y, ssq);
          ssq = __fmaf_rn(x.z, x.z, ssq);
          ssq = __fmaf_rn(x.w, x.w, ssq);
        }
      }
    }
  }
  return ssq;
}

// Local hand-off (tag_in): the previous phase's output vector, polled in place.
template <int UP>
__device__ __forceinline__ void stage_handoff_inline(const unsigned long long* src, unsigned tag, int n4, int t, int NT,
                                                     float4* xs4) {
  const long long t_start = clock64();
  for (int pb = t; pb < n4; pb += NT * UP) {
    unsigned long long wd[UP][4];  // every slot loads (clamped index): keeps the buffer in registers, see stage_exchange
    bool ok;
    unsigned seen = tag;
    do {
      ok = true;
#pragma unroll
      for (int k = 0; k < UP; ++k) {
        const int p = min(pb + k * NT, n4 - 1);
        ld_tagged2_gpu(src + 4 * p, wd[k][0], wd[k][1]);
        ld_tagged2_gpu(src + 4 * p + 2, wd[k][2], wd[k][3]);
      }
#pragma unroll
      for (int k = 0; k < UP; ++k)
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (tag_of(wd[k][e]) != tag) {
            ok = false;
            seen = tag_of(wd[k][e]);
          }
      if (!ok) poll_failed(seen, tag, t_start, 2);
    } while (!ok);
#pragma unroll
    for (int k = 0; k < UP; ++k) {
      const int p = pb + k * NT;
      if (p < n4) xs4[p] = make_float4(val_of(wd[k][0]), val_of(wd[k][1]), val_of(wd[k][2]), val_of(wd[k][3]));
    }
  }
}
template <int UP>
__device__ KLLM_STAGE_CALL void stage_handoff(const unsigned long long* src, unsigned tag, int n4, int t, int NT,
                                              float4* xs4) {
  stage_handoff_inline<UP>(src, tag, n4, t, NT, xs4);
}

// ---- one GEMV phase of one CTA's consumer warps --------------------------------------------------
// Stages the phase's input vector (tagged residual exchange / tagged hand-off / plain vector) into
// shared memory, RMS-normalises it when the phase asks for it, consumes this CTA's ring stages
// task by task, runs the epilogues and, for the classifier, leaves the CTA's (max, index).
template <int CW, bool INT8, bool PROF>
__device__ KLLM_PHASE_CALL Carry gemv_phase(const Params& P, Carry carry, int tok, int pos, const float* emb_row,
                                            unsigned long long* stamp) {
  constexpr int CT = CW * 32;
  constexpr int wbytes = INT8 ? 1 : 4;
  const Phase& ph = g_ph_cons;
  uint64_t* full_bar = g_full_bar;
  uint64_t* empty_bar = g_empty_bar;
  float* s_warp = g_s_warp;
  float* s_argv = g_s_argv;
  int* s_argi = g_s_argi;
  float* xs = reinterpret_cast<float*>(smem + kCtlBytes);                  // phase input vector
  float* xres = reinterpret_cast<float*>(smem + kCtlBytes + P.xbuf_bytes);  // residual stream (tagged modes)
  unsigned char* stages = smem + kCtlBytes + P.xbuf_bytes + P.xres_bytes;
  float4* xs4w = reinterpret_cast<float4*>(xs);
  float4* xres4 = reinterpret_cast<float4*>(xres);
  const float4* xs4 = reinterpret_cast<const float4*>(xs);
  const int S = P.num_stages;
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const int cta = blockIdx.x;
  const int G = gridDim.x;
  Pipe pipe = carry.pipe;
  ArgBest best{carry.best_v, carry.best_i};
  if (!PROF) stamp = nullptr;
  auto hand_tag = [&](int hand) {
    return P.hand_base + static_cast<unsigned>(tok * P.hands_per_token + hand) + 1u;
  };

  // ---- stage the input vector (and RMS-normalise it) --------------------------------------
  const int M = ph.in_dim;
  const int n4 = M >> 2;
  const bool has_norm = ph.norm_w != nullptr;
  float ssq = 0.f;
  bool ssq_ready = false;
  // The RMSNorm weight of the phase does not depend on anything: fetch this thread's packs from L2
  // BEFORE polling the input, so their latency (~0.4 us) hides behind the poll instead of following it.
  // Fat-warp builds only (the thin int8 build has no registers to park them in); vectors too long for
  // kNormPre packs per thread are read after the poll as before.  Slots past the end re-read the last
  // pack so that the buffer is always written (stays in registers).
  constexpr int kNormPre = CW <= 6 ? 3 : (CW <= 8 ? 2 : 0);
  const bool norm_pre = kNormPre > 0 && has_norm && n4 <= kNormPre * CT;
  float4 nw_pre[kNormPre > 0 ? kNormPre : 1];
  if (kNormPre > 0 && norm_pre) {
    const float4* nw4 = reinterpret_cast<const float4*>(ph.norm_w);
#pragma unroll
    for (int k = 0; k < kNormPre; ++k) nw_pre[k] = __ldg(nw4 + min(tid + k * CT, n4 - 1));
  } else {
#pragma unroll
    for (int k = 0; k < (kNormPre > 0 ? kNormPre : 1); ++k) nw_pre[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  if (ph.tp_in) {
    // x = x_old + (p_0 + ... + p_{W-1}); no grid barrier, no all-reduce kernel
    const unsigned tag = P.tp_seq_base + static_cast<unsigned>(tok * P.exch_per_token + ph.exch) + 1u;
    const unsigned long long* area =
        P.tp_data[P.tp_rank] + static_cast<size_t>(tag & 1u) * P.tp_world * P.tp_stride;
    switch (P.tp_world) {
      case 1:
        // Many thin warps (int8 build, 96 registers): all threads poll two packs each -- the poll
        // buffers of a deeper batch would spill, and a spill is an L2 round trip here; the sum of
        // squares is then taken from shared memory.  Few fat warps: the 128 rmsnorm threads poll four
        // packs each and fold the sum of squares into the same pass.
        if (CW >= 12) {
          stage_exchange<1, 2, false>(area, P.tp_stride, tag, n4, tid, CT, xs4w, xres4);
        } else if (has_norm) {
          if (tid < kNormThreads)
            ssq = stage_exchange<1, 4, true>(area, P.tp_stride, tag, n4, tid, kNormThreads, xs4w, xres4);
          ssq_ready = true;
        } else {
          stage_exchange<1, 4, false>(area, P.tp_stride, tag, n4, tid, CT, xs4w, xres4);
        }
        break;
      case 2: stage_exchange<2, 2, false>(area, P.tp_stride, tag, n4, tid, CT, xs4w, xres4); break;
      case 4: stage_exchange<4, 1, false>(area, P.tp_stride, tag, n4, tid, CT, xs4w, xres4); break;
      default: stage_exchange<8, 1, false>(area, P.tp_stride, tag, n4, tid, CT, xs4w, xres4); break;
    }
  } else if (ph.tag_in != nullptr) {
    if (CW >= 12)
      stage_handoff<2>(ph.tag_in, hand_tag(ph.hand_in), n4, tid, CT, xs4w);
    else
      stage_handoff<4>(ph.tag_in, hand_tag(ph.hand_in), n4, tid, CT, xs4w);
  } else {
    const float4* xg4 = reinterpret_cast<const float4*>(ph.x_from_emb ? emb_row : ph.x);
    for (int i = tid; i < n4; i += CT) xs4w[i] = __ldcg(xg4 + i);
  }
  if (stamp) stamp[10] = global_ns();
  if (has_norm) {
    // rmsnorm_kernel.cu:4-50: 128 threads, thread t sums the squares of packs t, t+128, ... with
    // one FFMA chain, cub<128> block reduction, rsqrt(mean + eps), then (scale * x) * w
    if (!ssq_ready) {
      consumer_sync<CT>();
      if (tid < kNormThreads)
        for (int p = tid; p < n4; p += kNormThreads) {
          const float4 v = xs4[p];
          ssq = __fmaf_rn(v.x, v.x, ssq);
          ssq = __fmaf_rn(v.y, v.y, ssq);
          ssq = __fmaf_rn(v.z, v.z, ssq);
          ssq = __fmaf_rn(v.w, v.w, ssq);
        }
    }
    if (tid < kNormThreads) {
      const float ws = warp_tree_sum(ssq);
      if (lane == 0) s_warp[warp] = ws;
    }
    consumer_sync<CT>();
    const float total = __fadd_rn(__fadd_rn(__fadd_rn(s_warp[0], s_warp[1]), s_warp[2]), s_warp[3]);
    const float sc = rsqrtf(__fadd_rn(__fdiv_rn(total, static_cast<float>(M)), ph.norm_eps));
    {
      // the norm weight (dim floats, the same for every CTA and token) comes from L2 here, once the
      // scale is known: keeping it in registers across the poll made ptxas spill, and with the ring
      // taking all of shared memory a spill is an L2 round trip too
      const float4* nw4 = reinterpret_cast<const float4*>(ph.norm_w);
      auto scale_pack = [&](int i, const float4& nw) {
        float4 v = xs4w[i];
        v.x = __fmul_rn(__fmul_rn(sc, v.x), nw.x);
        v.y = __fmul_rn(__fmul_rn(sc, v.y), nw.y);
        v.z = __fmul_rn(__fmul_rn(sc, v.z), nw.z);
        v.w = __fmul_rn(__fmul_rn(sc, v.w), nw.w);
        xs4w[i] = v;
      };
      if (kNormPre > 0 && norm_pre) {
#pragma unroll
        for (int k = 0; k < kNormPre; ++k)
          if (tid + k * CT < n4) scale_pack(tid + k * CT, nw_pre[k]);
      } else {
        for (int i = tid; i < n4; i += CT) scale_pack(i, __ldg(nw4 + i));
      }
    }
  }
  consumer_sync<CT>();
  // int8 fast mode: the staged (and normalised) vector becomes 24-bit fixed point per 64-group
  const bool int8_fast = INT8 && P.int8_fast != 0 && ph.group_size == 64 && (M & 63) == 0;
  if constexpr (INT8) {
    if (int8_fast) quantize_input_inplace<CT>(xs, M, tid);
  }
  if (stamp) stamp[1] = global_ns();

  const int u0 = static_cast<int>(static_cast<long long>(cta) * ph.units / G);
  const int u1 = static_cast<int>(static_cast<long long>(cta + 1) * ph.units / G);
  const int rpu = ph.swiglu ? 2 : 1;
  const int row_bytes = M * wbytes;
  const float* residual = ph.residual_from_emb ? emb_row : ph.residual;

  // bias / residual of a row are fetched BEFORE its dot product so their L2 latency hides
  // behind the accumulation (by the lane that will run the row's epilogue)
  auto prefetch_addend = [&](int unit, float& bias_v, float& res_v) {
    bias_v = 0.f, res_v = 0.f;
    if (ph.swiglu) return;
    const RowRef rr = resolve_row(ph, unit, 0);
    if (ph.seg[rr.seg].bias != nullptr) bias_v = __ldg(ph.seg[rr.seg].bias + rr.row);
    if (residual != nullptr) res_v = __ldcg(residual + rr.row);
  };
  // one lane per unit
  auto epilogue = [&](int unit, float d0, float d1, float bias_v, float res_v) {
    if (ph.swiglu) {
      const float g = swiglu_ref(d0, d1);
      if (ph.seg[0].tag_out != nullptr)
        st_tagged_gpu(ph.seg[0].tag_out + unit, g, hand_tag(ph.hand_out));
      else
        ph.seg[0].out[unit] = g;
      return;
    }
    if (ph.tp_out) {
      const unsigned tag = P.tp_seq_base + static_cast<unsigned>(tok * P.exch_per_token + ph.exch_out) + 1u;
      const size_t off = (static_cast<size_t>(tag & 1u) * P.tp_world + P.tp_rank) * P.tp_stride + unit;
      if (P.tp_world == 1) {
        st_tagged_gpu(P.tp_data[0] + off, d0, tag);
      } else {
        for (int k = 1; k <= P.tp_world; ++k) st_tagged(P.tp_data[(P.tp_rank + k) % P.tp_world] + off, d0, tag);
      }
      return;
    }
    const RowRef rr = resolve_row(ph, unit, 0);
    const Seg& sg = ph.seg[rr.seg];
    float v = d0;
    if (sg.bias != nullptr) v = __fadd_rn(v, bias_v);       // matmul.cpp:74-77: out + bias
    if (residual != nullptr) v = __fadd_rn(res_v, v);       // llama3.cpp:683,719: x + out
    if (sg.tag_out != nullptr) st_tagged_gpu(sg.tag_out + rr.row, v, hand_tag(ph.hand_out));
    if (sg.out == nullptr) {
    } else if (sg.head_major) {  // value cache [kv_head][SP][seq_len][dv]
      const int hs = P.head_size, dv = hs / P.attn_vsplit;
      const int kvh = rr.row / hs, d = rr.row % hs;
      sg.out[((static_cast<size_t>(kvh) * P.attn_vsplit + d / dv) * P.seq_len + pos) * dv + d % dv] = v;
    } else {
      sg.out[static_cast<long long>(pos) * sg.pos_stride + rr.row] = v;
    }
    if (ph.argmax) arg_fold(best, v, rr.row);
  };

  long long cyc_wait = 0, cyc_rows = 0;
  long long cyc4[4] = {0, 0, 0, 0};
  if (ph.chunks_per_row == 1) {
    // A stage holds n units; they are handed out as tasks of up to 4 rows (plain: 4 units, SwiGLU:
    // 2 units = w1 + w3 rows of two outputs), task after task round-robin over the consumer warps.
    const int ups = ph.rows_per_stage / rpu;
    // Rows per task (compile-time knob KLLM_TASK_ROWS: 1, 2 or 4).  A CTA owns only 14-83 rows of a
    // phase and every consumer warp has to pass (wait + arrive) every ring stage in order, so a warp
    // sitting on a fat task while its neighbours have none holds up the refill of the whole ring.
    // The host picks the rows per task of each phase (MegaEngine::init, pick_task_rows): short phases
    // whose rows are already in the ring when they start are as slow as their slowest warp, so they
    // want many small tasks; long ones want fat tasks that share the loads of the input vector.
    constexpr int kTaskRows = KLLM_TASK_ROWS;  // upper bound (compile time: which dot_rows<> forms exist)
    const int task_rows = min(kTaskRows, max(1, ph.task_rows));
    const int upt = ph.swiglu ? (task_rows >= 2 ? task_rows / 2 : 1) : task_rows;  // units per task
    int task = 0;                      // tasks of this phase so far (same count in every warp)
    for (int u = u0; u < u1; u += ups) {
      const int n = min(ups, u1 - u);
      const long long c0 = stamp ? clock64() : 0;
      mbar_wait(&full_bar[pipe.slot], pipe.parity);
      const long long c1 = stamp ? clock64() : 0;
      cyc_wait += c1 - c0;
      const unsigned char* sbase = stages + static_cast<size_t>(pipe.slot) * P.stage_bytes;
      if constexpr (INT8) {
        if (ph.team && int8_fast) {
          // TEAM form.  With one task per warp the (six) stages of the ring are consumed side by side and
          // released together: the producer cannot refill while the consumers compute, and a phase takes the
          // sum of both (measured: int8 rows at half the HBM rate).  Here kTeam warps share ONE stage -- each
          // takes a slice of the columns of all its rows -- so stages are finished and released one after the
          // other and the refill of the first overlaps the arithmetic on the next.  Member 0 adds the members'
          // row partials (in member order, through shared memory) and runs the epilogues.
          constexpr int kTeam = (CW % 4 == 0) ? 4 : 2, kTeams = CW / kTeam;
          const int team = warp / kTeam, member = warp % kTeam;
          if (task % kTeams == team) {
            const int j = lane >> 2;  // lane 4 j ends with the total of stage row j
            const bool owner = member == 0 && (lane & 3) == 0 && j < n;
            float bias_v = 0.f, res_v = 0.f;
            if (owner) prefetch_addend(u + j, bias_v, res_v);
            const int nrows = n * rpu;
            float tot = 0.f;
            if (ph.mma) {  // <= 8 rows on the tensor cores; the member's share of the 64-element groups
              const uint32_t pad = static_cast<uint32_t>(ph.row_pad);
              const int groups = M >> 6;
              tot = accum_w8_mma(smem_u32(sbase), static_cast<uint32_t>(row_bytes) + pad,
                                 smem_u32(sbase) + static_cast<uint32_t>(ph.scale_off),
                                 static_cast<uint32_t>(ph.scale_row_bytes) + pad, nrows, smem_u32(xs),
                                 groups * member / kTeam, groups * (member + 1) / kTeam, lane);
            } else {  // one or two long rows on dp4a; the member's share of the 512-element steps
              const int steps = (M + 511) >> 9;
              const uint32_t wa = smem_u32(sbase), sa = wa + static_cast<uint32_t>(ph.scale_off);
              const uint32_t w2[2] = {wa, wa + (nrows > 1 ? static_cast<uint32_t>(row_bytes) : 0u)};
              const uint32_t s2[2] = {sa, sa + (nrows > 1 ? static_cast<uint32_t>(ph.scale_row_bytes) : 0u)};
              float a2[2] = {0.f, 0.f};
              accum_w8_dp4a<2>(w2, s2, smem_u32(xs), M, lane, a2, steps * member / kTeam, steps * (member + 1) / kTeam);
#pragma unroll
              for (int off = 16; off > 0; off >>= 1) {
                a2[0] += __shfl_xor_sync(kFull, a2[0], off);
                a2[1] += __shfl_xor_sync(kFull, a2[1], off);
              }
              tot = j == 0 ? a2[0] : a2[1];
            }
            float* scratch = &g_s_team[team][(task / kTeams) & 1][0][0];
            if (member != 0 && (lane & 3) == 0) scratch[(member - 1) * 8 + j] = tot;
            asm volatile("bar.sync %0, %1;" ::"r"(2 + team), "n"(kTeam * 32) : "memory");  // the warps of the team
            if (member == 0) {
#pragma unroll
              for (int mm = 1; mm < kTeam; ++mm) tot = __fadd_rn(tot, scratch[(mm - 1) * 8 + j]);
              // SwiGLU stage order: w1 rows of the n units, then their w3 rows
              const float tot_w3 = __shfl_sync(kFull, tot, min(j + n, 7) * 4);
              if (owner) epilogue(u + j, tot, tot_w3, bias_v, res_v);
            }
          }
          ++task;
          __syncwarp();
          if (stamp) cyc_rows += clock64() - c1;
          if (lane == 0) mbar_arrive(&empty_bar[pipe.slot]);
          pipe.advance(S);
          continue;
        }
      }
      for (int i0 = 0; i0 < n; i0 += upt, ++task) {
        if (task % CW != warp) continue;  // CW is 6, 8 or 16: a real modulo (a mask would idle warps 2 and 3 of 6)
        const int nu = min(upt, n - i0);
        const long long t_a = stamp ? clock64() : 0;
        float bias_v = 0.f, res_v = 0.f;
        if (lane < nu) prefetch_addend(u + i0 + lane, bias_v, res_v);
        const long long t_b = stamp ? clock64() : 0;
        float e0 = 0.f, e1 = 0.f;  // this lane's unit: its dot product(s)
        // shared-window addresses of the stage's rows / scale rows
        const uint32_t rb = static_cast<uint32_t>(row_bytes), srb = static_cast<uint32_t>(ph.scale_row_bytes);
        const uint32_t wa = smem_u32(sbase), sa = smem_u32(sbase) + static_cast<uint32_t>(ph.scale_off);
        const uint32_t xa = smem_u32(xs);
        if (ph.swiglu) {
          // stage order: w1 rows of the n units, then their w3 rows
          if (kTaskRows == 4 && nu == 2) {
            const Rows4 rp{{wa + i0 * rb, wa + (n + i0) * rb, wa + (i0 + 1) * rb, wa + (n + i0 + 1) * rb}};
            const Rows4 sp{{sa + i0 * srb, sa + (n + i0) * srb, sa + (i0 + 1) * srb, sa + (n + i0 + 1) * srb}};
            const float4 d = dot_rows<4, INT8>(rp, sp, xa, M, ph.group_size, ph.group_shift, lane, int8_fast);
            e0 = lane == 0 ? d.x : d.z;
            e1 = lane == 0 ? d.y : d.w;
          } else {
            const Rows4 rp{{wa + i0 * rb, wa + (n + i0) * rb, 0u, 0u}};
            const Rows4 sp{{sa + i0 * srb, sa + (n + i0) * srb, 0u, 0u}};
            const float4 d = dot_rows<2, INT8>(rp, sp, xa, M, ph.group_size, ph.group_shift, lane, int8_fast);
            e0 = d.x, e1 = d.y;
          }
        } else if (kTaskRows == 4 && nu == 4) {
          const Rows4 rp{{wa + i0 * rb, wa + (i0 + 1) * rb, wa + (i0 + 2) * rb, wa + (i0 + 3) * rb}};
          const Rows4 sp{{sa + i0 * srb, sa + (i0 + 1) * srb, sa + (i0 + 2) * srb, sa + (i0 + 3) * srb}};
          const float4 d = dot_rows<4, INT8>(rp, sp, xa, M, ph.group_size, ph.group_shift, lane, int8_fast);
          e0 = lane == 0 ? d.x : lane == 1 ? d.y : lane == 2 ? d.z : d.w;
        } else {
          int r0 = 0;
          if (nu >= 2) {
            const Rows4 rp{{wa + i0 * rb, wa + (i0 + 1) * rb, 0u, 0u}};
            const Rows4 sp{{sa + i0 * srb, sa + (i0 + 1) * srb, 0u, 0u}};
            const float4 d = dot_rows<2, INT8>(rp, sp, xa, M, ph.group_size, ph.group_shift, lane, int8_fast);
            e0 = lane == 0 ? d.x : d.y;
            r0 = 2;
          }
          if (r0 < nu) {  // nu is 1 or 3: one more row
            const Rows4 rp{{wa + (i0 + r0) * rb, 0u, 0u, 0u}};
            const Rows4 sp{{sa + (i0 + r0) * srb, 0u, 0u, 0u}};
            const float4 d = dot_rows<1, INT8>(rp, sp, xa, M, ph.group_size, ph.group_shift, lane, int8_fast);
            if (lane == r0) e0 = d.x;
          }
        }
        const long long t_c = stamp ? clock64() : 0;
        if (lane < nu) epilogue(u + i0 + lane, e0, e1, bias_v, res_v);
        if (stamp) {
          cyc4[0] += t_b - t_a, cyc4[1] += t_c - t_b, cyc4[3] += clock64() - t_c;
        }
      }
      __syncwarp();
      if (stamp) cyc_rows += clock64() - c1;
      if (lane == 0) mbar_arrive(&empty_bar[pipe.slot]);
      pipe.advance(S);
    }
  } else {
    // rows longer than a stage (fp32 only): the owning warp carries its partial sums across
    // consecutive stages; chunk boundaries are multiples of 128 packs so every virtual
    // thread still sees its packs in increasing order.
    for (int u = u0; u < u1; ++u) {
      const bool mine = (u - u0) % CW == warp;
      float bias_v = 0.f, res_v = 0.f;
      if (mine && lane == 0) prefetch_addend(u, bias_v, res_v);
      float acc[1][4] = {{0.f, 0.f, 0.f, 0.f}};
      for (int c = 0; c < ph.chunks_per_row; ++c) {
        const int e0 = c * ph.chunk_elems;
        const int ne = min(ph.chunk_elems, M - e0);
        mbar_wait(&full_bar[pipe.slot], pipe.parity);
        if (mine) {
          const uint32_t w[1] = {smem_u32(stages + static_cast<size_t>(pipe.slot) * P.stage_bytes)};
          accum_f32<1>(w, smem_u32(xs) + static_cast<uint32_t>(e0) * 4u, ne >> 2, lane, acc);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[pipe.slot]);
        pipe.advance(S);
      }
      if (mine) {
        const float d0 = block128_sum_vt_packed(acc[0], lane);
        if (lane == 0) epilogue(u, d0, 0.f, bias_v, res_v);
      }
    }
  }

  if (ph.argmax) {
    // per-CTA (max, lowest index) of the classifier rows this CTA produced: the (up to four) lanes
    // that ran epilogues hold partial bests
    ArgBest wb = best;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {  // (the mma form runs its epilogues in lanes 0, 4, ..., 28)
      const float ov = __shfl_xor_sync(kFull, wb.v, off);
      const int oi = __shfl_xor_sync(kFull, wb.i, off);
      arg_fold(wb, ov, oi);
    }
    if (lane == 0) {
      s_argv[warp] = wb.v;
      s_argi[warp] = wb.i;
    }
    consumer_sync<CT>();
    if (tid == 0) {
      ArgBest b{0.f, -1};
      for (int w = 0; w < CW; ++w) arg_fold(b, s_argv[w], s_argi[w]);
      P.arg_val[cta] = b.v;
      P.arg_idx[cta] = b.i;
    }
  }
  if (stamp) {
    stamp[2] = global_ns();
    stamp[4] = static_cast<unsigned long long>(cyc4[0]);
    stamp[5] = static_cast<unsigned long long>(cyc4[1]);
    stamp[6] = static_cast<unsigned long long>(cyc4[2]);
    stamp[7] = static_cast<unsigned long long>(cyc4[3]);
    stamp[8] = static_cast<unsigned long long>(cyc_wait);
    stamp[9] = static_cast<unsigned long long>(cyc_rows);
  }
  return Carry{pipe, best.v, best.i};
}

// ---- tensor parallel, classifier sharded by vocabulary ----------------------------------------------
// Rank r computed logits rows [r V/W, (r+1) V/W) and published them as tagged words into EVERY rank's
// exchange area (the tp_out epilogue, exchange `ph.exch`).  Here the CTAs of this rank split the V
// words of the local area between them: poll, store the logit, keep (max, lowest index).  All ranks
// end with the same full logits vector and the same per-CTA partials, hence the same greedy id --
// the cross-rank argmax needs no further exchange.
template <int CW>
__device__ __noinline__ void gather_logits_phase(const Params& P, int tok) {
  constexpr int CT = CW * 32;
  const Phase& ph = g_ph_cons;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int cta = blockIdx.x, G = gridDim.x;
  const int V = ph.units, rows = ph.in_dim;  // rows per rank
  const unsigned tag = P.tp_seq_base + static_cast<unsigned>(tok * P.exch_per_token + ph.exch) + 1u;
  const unsigned long long* area =
      P.tp_data[P.tp_rank] + static_cast<size_t>(tag & 1u) * P.tp_world * P.tp_stride;
  const int u0 = static_cast<int>(static_cast<long long>(cta) * V / G);
  const int u1 = static_cast<int>(static_cast<long long>(cta + 1) * V / G);
  float* logits = ph.seg[0].out;
  ArgBest best{0.f, -1};
  for (int i = u0 + tid; i < u1; i += CT) {
    const int r = i / rows, j = i - r * rows;
    const float v = poll_tagged_sys(area + static_cast<size_t>(r) * P.tp_stride + j, tag);
    logits[i] = v;
    arg_fold(best, v, i);
  }
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const float ov = __shfl_xor_sync(kFull, best.v, off);
    const int oi = __shfl_xor_sync(kFull, best.i, off);
    arg_fold(best, ov, oi);
  }
  if (lane == 0) {
    g_s_argv[warp] = best.v;
    g_s_argi[warp] = best.i;
  }
  consumer_sync<CT>();
  if (tid == 0) {
    ArgBest b{0.f, -1};
    for (int w = 0; w < CW; ++w) arg_fold(b, g_s_argv[w], g_s_argi[w]);
    P.arg_val[cta] = b.v;
    P.arg_idx[cta] = b.i;
  }
}

// ---- the kernel ---------------------------------------------------------------------------------
template <int CW, bool INT8, bool PROF>
__global__ void __launch_bounds__(CW * 32 + 64, 1) decode_megakernel(const __grid_constant__ Params P) {
  constexpr int CT = CW * 32;  // consumer threads
  uint64_t* full_bar = g_full_bar;
  uint64_t* empty_bar = g_empty_bar;
  Phase& s_phase_cons = g_ph_cons;
  Phase& s_phase_prod = g_ph_prod;
  Phase& s_phase_pf = g_ph_pf;
  volatile unsigned& s_fill_count = g_fill_count;

  float* xres = reinterpret_cast<float*>(smem + kCtlBytes + P.xbuf_bytes);  // residual stream (tagged modes)
  unsigned char* stages = smem + kCtlBytes + P.xbuf_bytes + P.xres_bytes;
  const int S = P.num_stages;
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const bool is_producer = warp == CW;
  const int cta = blockIdx.x;
  const int G = gridDim.x;

  if (tid == 0) {
    s_fill_count = 0u;
    for (int s = 0; s < S; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], CW);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  Pipe pipe{0, 0u};
  constexpr int wbytes = INT8 ? 1 : 4;

  // =============================== producer warp ===============================================
  if (is_producer) {
    const uint64_t policy = policy_evict_first();  // weights: streamed once per token
    const uint64_t policy_kv = policy_evict_last();  // KV tiles: re-read every token, keep in L2
    unsigned filled = 0u;
    int ppos = P.state->pos;
    for (int tok = 0; tok < P.n_tokens; ++tok, ++ppos) {
      const int n_run = tok < P.skip_cls_tokens ? P.n_phases - P.n_cls_phases : P.n_phases;  // prompt token: no classifier
      for (int pi = 0; pi < n_run; ++pi) {
        {
          const uint32_t* src = reinterpret_cast<const uint32_t*>(P.phases + pi);
          uint32_t* dst = reinterpret_cast<uint32_t*>(&s_phase_prod);
          __syncwarp();
          for (int i = lane; i < static_cast<int>(sizeof(Phase) / 4); i += 32) dst[i] = __ldg(src + i);
          __syncwarp();
        }
        const Phase& ph = s_phase_prod;
        if (ph.kind == kPhaseGather) continue;  // nothing to stream
        if (ph.kind != kPhaseGemv) {
          const int SP = P.attn_split;
          if (cta >= P.head_num * SP || ppos == 0) continue;
          // rows t < pos of this head: final since the previous token.  Order the async-proxy
          // reads after the grid barrier that closed the previous token.
          if (tok > 0 && lane == 0) {
            const unsigned need = P.barrier_base +
                                  static_cast<unsigned>((tok - 1) * P.bars_per_token + ph.barrier_idx) *
                                      static_cast<unsigned>(G);
            while (static_cast<int>(ld_acquire_u32(P.barrier) - need) < 0) {
            }
            asm volatile("fence.proxy.async;" ::: "memory");
          }
          __syncwarp();
          const int hs = P.head_size;
          const int head = cta / SP, split = cta % SP;
          const int kvh = head / P.kv_mul;
          const size_t head_block =
              (static_cast<size_t>(ph.layer) * (P.kv_dim / hs) + kvh) * P.seq_len * hs;
          if (ph.kind == kPhaseAttnFlash) {  // tiles j = split, split + SP, ...: K tile, then V tile
            const int T = P.attn_tile;
            const float* kbase = P.key_cache + head_block;
            const float* vbase = P.value_cache + head_block;
            const int n_tiles = attn_tiles(ppos, T);
            for (int j = split; j < n_tiles; j += SP) {
              const int t0 = j * T;
              const int nt = min(T, ppos - t0);
              for (int kv = 0; kv < 2; ++kv) {
                mbar_wait(&empty_bar[pipe.slot], pipe.parity ^ 1u);
                unsigned char* dst = stages + static_cast<size_t>(pipe.slot) * P.stage_bytes;
                if (lane == 0) mbar_expect_tx(&full_bar[pipe.slot], static_cast<uint32_t>(nt) * hs * 4);
                __syncwarp();
                if (kv == 0) {
                  if (lane < (hs >> 2))
                    bulk_g2s(dst + static_cast<size_t>(lane) * T * 16,
                             kbase + (static_cast<size_t>(lane) * P.seq_len + t0) * 4,
                             static_cast<uint32_t>(nt) * 16, &full_bar[pipe.slot], policy_kv);
                } else if (lane == 0) {
                  bulk_g2s(dst, vbase + static_cast<size_t>(t0) * hs, static_cast<uint32_t>(nt) * hs * 4,
                           &full_bar[pipe.slot], policy_kv);
                }
                pipe.advance(S);
                if (lane == 0) s_fill_count = ++filled; else ++filled;
              }
            }
            continue;
          }
          if (ph.kind != kPhaseAttnPV) {  // K tiles j = split, split + SP, ... (fused: SP == 1, all of them)
            const int T = P.attn_tile;
            const float* kbase = P.key_cache + head_block;
            const int n_tiles = attn_tiles(ppos, T);
            for (int j = split; j < n_tiles; j += SP) {
              const int t0 = j * T;
              const int nt = min(T, ppos - t0);
              mbar_wait(&empty_bar[pipe.slot], pipe.parity ^ 1u);
              unsigned char* dst = stages + static_cast<size_t>(pipe.slot) * P.stage_bytes;
              if (lane == 0) mbar_expect_tx(&full_bar[pipe.slot], static_cast<uint32_t>(nt) * hs * 4);
              __syncwarp();
              if (lane < (hs >> 2))  // hs <= 128 (checked on the host): one 16-byte chunk column per lane
                bulk_g2s(dst + static_cast<size_t>(lane) * T * 16,
                         kbase + (static_cast<size_t>(lane) * P.seq_len + t0) * 4,
                         static_cast<uint32_t>(nt) * 16, &full_bar[pipe.slot], policy_kv);
              pipe.advance(S);
              if (lane == 0) s_fill_count = ++filled; else ++filled;
            }
          }
          if (ph.kind != kPhaseAttention) {  // this CTA's slice of V: [seq_len][dv] contiguous
            const int dv = hs / SP, T = P.attn_tile_v;
            const float* vbase = P.value_cache + head_block + static_cast<size_t>(split) * P.seq_len * dv;
            const int n_tiles = attn_tiles(ppos, T);
            for (int j = 0; j < n_tiles; ++j) {
              const int t0 = j * T;
              const int nt = min(T, ppos - t0);
              mbar_wait(&empty_bar[pipe.slot], pipe.parity ^ 1u);
              unsigned char* dst = stages + static_cast<size_t>(pipe.slot) * P.stage_bytes;
              if (lane == 0) {
                mbar_expect_tx(&full_bar[pipe.slot], static_cast<uint32_t>(nt) * dv * 4);
                bulk_g2s(dst, vbase + static_cast<size_t>(t0) * dv, static_cast<uint32_t>(nt) * dv * 4,
                         &full_bar[pipe.slot], policy_kv);
              }
              __syncwarp();
              pipe.advance(S);
              if (lane == 0) s_fill_count = ++filled; else ++filled;
            }
          }
          continue;
        }
        const int u0 = static_cast<int>(static_cast<long long>(cta) * ph.units / G);
        const int u1 = static_cast<int>(static_cast<long long>(cta + 1) * ph.units / G);
        const int rpu = ph.swiglu ? 2 : 1;
        const int row_bytes = ph.in_dim * wbytes;
        if (ph.chunks_per_row == 1) {
          const int ups = ph.rows_per_stage / rpu;
          for (int u = u0; u < u1; u += ups) {
            const int n = min(ups, u1 - u);
            const int nrows = n * rpu;
            mbar_wait(&empty_bar[pipe.slot], pipe.parity ^ 1u);
            unsigned char* dst = stages + static_cast<size_t>(pipe.slot) * P.stage_bytes;
            if (lane == 0)
              mbar_expect_tx(&full_bar[pipe.slot],
                             static_cast<uint32_t>(nrows) * (row_bytes + ph.scale_row_bytes));
            __syncwarp();
            if (ph.row_pad) {
              // padded rows (mma form, nrows <= 8): one copy per weight row (lanes 0..7) and per scale row (16..23)
              const int j = lane & 15;
              if (j < nrows && (lane & 8) == 0) {
                const RowRef rr = stage_row(ph, u, n, j);
                const long long e = static_cast<long long>(rr.row) * ph.in_dim;
                if (lane < 16) {
                  bulk_g2s(dst + static_cast<size_t>(j) * (row_bytes + ph.row_pad),
                           static_cast<const unsigned char*>(ph.seg[rr.seg].w) + e * wbytes, static_cast<uint32_t>(row_bytes),
                           &full_bar[pipe.slot], policy);
                } else {
                  const long long g0 = ph.group_shift >= 0 ? (e >> ph.group_shift) : (e / ph.group_size);
                  bulk_g2s(dst + ph.scale_off + static_cast<size_t>(j) * (ph.scale_row_bytes + ph.row_pad),
                           ph.seg[rr.seg].scales + g0, static_cast<uint32_t>(ph.scale_row_bytes), &full_bar[pipe.slot],
                           policy);
                }
              }
            } else {  // one bulk copy per run of consecutive rows of one matrix (nrows <= 32: lane = row)
              const RowRef rr = lane < nrows ? stage_row(ph, u, n, lane) : RowRef{-1, -1};
              const int len = run_length(rr, lane, nrows);
              if (len > 0) {
                const long long e = static_cast<long long>(rr.row) * ph.in_dim;
                const unsigned char* src = static_cast<const unsigned char*>(ph.seg[rr.seg].w) + e * wbytes;
                bulk_g2s(dst + static_cast<size_t>(lane) * row_bytes, src, static_cast<uint32_t>(len) * row_bytes,
                         &full_bar[pipe.slot], policy);
                if (ph.scale_row_bytes) {
                  const long long g0 = ph.group_shift >= 0 ? (e >> ph.group_shift) : (e / ph.group_size);
                  bulk_g2s(dst + ph.scale_off + static_cast<size_t>(lane) * ph.scale_row_bytes,
                           ph.seg[rr.seg].scales + g0, static_cast<uint32_t>(len) * ph.scale_row_bytes,
                           &full_bar[pipe.slot], policy);
                }
              }
            }
            pipe.advance(S);
            if (lane == 0) s_fill_count = ++filled; else ++filled;
          }
        } else {
          for (int u = u0; u < u1; ++u) {
            const RowRef rr = resolve_row(ph, u, 0);
            const unsigned char* src = static_cast<const unsigned char*>(ph.seg[rr.seg].w) +
                                       static_cast<long long>(rr.row) * row_bytes;
            for (int c = 0; c < ph.chunks_per_row; ++c) {
              const int e0 = c * ph.chunk_elems;
              const int ne = min(ph.chunk_elems, ph.in_dim - e0);
              mbar_wait(&empty_bar[pipe.slot], pipe.parity ^ 1u);
              if (lane == 0) {
                mbar_expect_tx(&full_bar[pipe.slot], static_cast<uint32_t>(ne) * wbytes);
                bulk_g2s(stages + static_cast<size_t>(pipe.slot) * P.stage_bytes,
                         src + static_cast<size_t>(e0) * wbytes, static_cast<uint32_t>(ne) * wbytes,
                         &full_bar[pipe.slot], policy);
              }
              __syncwarp();
              pipe.advance(S);
              if (lane == 0) s_fill_count = ++filled; else ++filled;
            }
          }
        }
      }
    }
    return;
  }

  // =============================== L2 prefetch warp ==============================================
  // The ring (num_stages x stage_bytes per SM, ~4 us of HBM time chip-wide) is shallower than the
  // dead time around a grid barrier or an attention phase, so HBM would idle there.  This warp
  // walks the same weight schedule as the producer, pf_stages ring-stages AHEAD of it, and only
  // pulls the bytes into L2 (cp.async.bulk.prefetch.L2): the outstanding window keeps HBM
  // streaming while the SMs wait for each other, and the ring then refills from L2.
  if (warp == CW + 1) {
    if (P.pf_stages <= 0) return;
    unsigned ahead = 0u;  // stages walked by this warp (same counting as the producer's `filled`)
    int ppos = P.state->pos;
    for (int tok = 0; tok < P.n_tokens; ++tok, ++ppos) {
      const int n_run = tok < P.skip_cls_tokens ? P.n_phases - P.n_cls_phases : P.n_phases;
      for (int pi = 0; pi < n_run; ++pi) {
        {
          const uint32_t* src = reinterpret_cast<const uint32_t*>(P.phases + pi);
          uint32_t* dst = reinterpret_cast<uint32_t*>(&s_phase_pf);
          __syncwarp();
          for (int i = lane; i < static_cast<int>(sizeof(Phase) / 4); i += 32) dst[i] = __ldg(src + i);
          __syncwarp();
        }
        const Phase& ph = s_phase_pf;
        if (ph.kind == kPhaseGather) continue;
        if (ph.kind != kPhaseGemv) {
          // KV tiles are L2-resident already (evict_last): count the producer's ring stages only
          if (cta < P.head_num * P.attn_split && ppos > 0) {
            if (ph.kind == kPhaseAttnFlash)
              ahead += 2u * static_cast<unsigned>(own_tiles(attn_tiles(ppos, P.attn_tile), cta % P.attn_split, P.attn_split));
            else if (ph.kind != kPhaseAttnPV)
              ahead += static_cast<unsigned>(own_tiles(attn_tiles(ppos, P.attn_tile), cta % P.attn_split, P.attn_split));
            if (ph.kind == kPhaseAttnPV || ph.kind == kPhaseAttnFused)
              ahead += static_cast<unsigned>(attn_tiles(ppos, P.attn_tile_v));
          }
          continue;
        }
        const int u0 = static_cast<int>(static_cast<long long>(cta) * ph.units / G);
        const int u1 = static_cast<int>(static_cast<long long>(cta + 1) * ph.units / G);
        const int rpu = ph.swiglu ? 2 : 1;
        const int row_bytes = ph.in_dim * wbytes;
        auto throttle = [&]() {
          while (static_cast<int>(ahead - s_fill_count) >= P.pf_stages) __nanosleep(400);
        };
        if (ph.chunks_per_row == 1) {
          const int ups = ph.rows_per_stage / rpu;
          for (int u = u0; u < u1; u += ups) {
            const int nrows = min(ups, u1 - u) * rpu;
            throttle();
            {
              const int n = nrows / rpu;
              const RowRef rr = lane < nrows ? stage_row(ph, u, n, lane) : RowRef{-1, -1};
              const int len = run_length(rr, lane, nrows);
              if (len > 0) {
                const long long e = static_cast<long long>(rr.row) * ph.in_dim;
                bulk_prefetch_l2(static_cast<const unsigned char*>(ph.seg[rr.seg].w) + e * wbytes,
                                 static_cast<uint32_t>(len) * row_bytes);
                if (ph.scale_row_bytes) {
                  const long long g0 = ph.group_shift >= 0 ? (e >> ph.group_shift) : (e / ph.group_size);
                  bulk_prefetch_l2(ph.seg[rr.seg].scales + g0, static_cast<uint32_t>(len) * ph.scale_row_bytes);
                }
              }
            }
            ++ahead;
          }
        } else {
          for (int u = u0; u < u1; ++u) {
            const RowRef rr = resolve_row(ph, u, 0);
            const unsigned char* src = static_cast<const unsigned char*>(ph.seg[rr.seg].w) +
                                       static_cast<long long>(rr.row) * row_bytes;
            for (int c = 0; c < ph.chunks_per_row; ++c) {
              const int e0 = c * ph.chunk_elems;
              const int ne = min(ph.chunk_elems, ph.in_dim - e0);
              throttle();
              if (lane == 0) bulk_prefetch_l2(src + static_cast<size_t>(e0) * wbytes, static_cast<uint32_t>(ne) * wbytes);
              ++ahead;
            }
          }
        }
      }
    }
    return;
  }

  // =============================== consumer warps ===============================================
  unsigned bar_target = P.barrier_base;
  int token = P.state->token;
  if (static_cast<unsigned>(token) >= static_cast<unsigned>(P.vocab_size)) token = 0;
  int pos = P.state->pos;
  int step = P.state->step;
  float4* xres4 = reinterpret_cast<float4*>(xres);
  constexpr int kPhaseWords = static_cast<int>(sizeof(Phase) / 4);
  static_assert(kPhaseWords <= CT, "phase copy: one word per consumer thread");
  uint32_t next_phase_word = tid < kPhaseWords ? __ldg(reinterpret_cast<const uint32_t*>(P.phases) + tid) : 0u;

  for (int tok = 0; tok < P.n_tokens; ++tok) {
    const float* emb_row = P.tok_emb + static_cast<size_t>(token) * P.dim;
    ArgBest best{0.f, -1};
    if (P.xres_bytes) {
      // the residual stream starts as the embedding row (llama3.cpp:578-598); the previous token's
      // last reader of xres (classifier staging) is behind the grid barrier that closed that token
      const float4* e4 = reinterpret_cast<const float4*>(emb_row);
      for (int i = tid; i < (P.dim >> 2); i += CT) xres4[i] = __ldg(e4 + i);
    }

    const bool prof_on = PROF && P.prof != nullptr && tok == P.prof_token && tid == 0;
    bool prev_barrier = true;
    auto hand_tag = [&](int hand) {
      return P.hand_base + static_cast<unsigned>(tok * P.hands_per_token + hand) + 1u;
    };
    for (int pi = 0; pi < P.n_phases; ++pi) {
      {
        // the grid barrier that ended the previous phase is the hazard fence for this copy; a
        // phase closed by a tagged exchange has none, so fence the CTA's own warps here
        if (!prev_barrier) consumer_sync<CT>();
        uint32_t* dst = reinterpret_cast<uint32_t*>(&s_phase_cons);
        if (tid < kPhaseWords) dst[tid] = next_phase_word;
        consumer_sync<CT>();
        // ... and the descriptor of the phase after this one starts its way from L2 now (one word per
        // thread), so that its latency hides behind this phase instead of opening the next
        const int npi = pi + 1 == P.n_phases ? 0 : pi + 1;
        if (tid < kPhaseWords) next_phase_word = __ldg(reinterpret_cast<const uint32_t*>(P.phases + npi) + tid);
      }
      const Phase& ph = s_phase_cons;
      unsigned long long* stamp =
          (PROF && prof_on) ? P.prof + (static_cast<size_t>(cta) * P.n_phases + pi) * kProfStamps : nullptr;
      if (stamp) stamp[0] = global_ns();

      if (ph.kind == kPhaseGather) {
        if (!(tok < P.skip_cls_tokens)) gather_logits_phase<CW>(P, tok);
        if (stamp) stamp[1] = stamp[2] = global_ns();
        if (ph.barrier_after) grid_barrier<CT>(P.barrier, bar_target, G);
        prev_barrier = ph.barrier_after != 0;
        if (stamp) stamp[3] = global_ns();
        continue;
      }
      if (ph.kind != kPhaseGemv) {
        const int SP = P.attn_split;
        if (cta < P.head_num * SP) {
          if (ph.kind == kPhaseAttnFlash)
            pipe = attention_flash_phase<CW>(P, cta / SP, cta % SP, pos, pipe, hand_tag(ph.hand_in), hand_tag(ph.hand_out), stamp);
          else if (ph.kind == kPhaseAttnFused)
            pipe = attention_fused_phase<CW>(P, cta, pos, pipe, hand_tag(ph.hand_in), hand_tag(ph.hand_out), stamp);
          else if (ph.kind == kPhaseAttention)
            pipe = attention_scores_phase<CW>(P, cta / SP, cta % SP, pos, pipe, hand_tag(ph.hand_in), hand_tag(ph.hand_out), stamp);
          else
            pipe = attention_pv_phase<CW>(P, cta / SP, cta % SP, pos, pipe, hand_tag(ph.hand_in), hand_tag(ph.hand_aux),
                                          hand_tag(ph.hand_out), stamp);
        }
        if (stamp) stamp[1] = stamp[2] = global_ns();
        if (ph.barrier_after) grid_barrier<CT>(P.barrier, bar_target, G);
        prev_barrier = ph.barrier_after != 0;
        if (stamp) stamp[3] = global_ns();
        continue;
      }
      prev_barrier = ph.barrier_after != 0;

      // A prompt token (llama3.cpp:733-745: predict(..., is_prompt = true) discards the logits and
      // returns -1) skips the classifier -- its weights are not even streamed -- but keeps the grid
      // barrier that closes the token.
      if (!(ph.cls && tok < P.skip_cls_tokens)) {
        const Carry out = gemv_phase<CW, INT8, PROF>(P, Carry{pipe, best.v, best.i}, tok, pos, emb_row, stamp);
        pipe = out.pipe;
        best.v = out.best_v, best.i = out.best_i;
      }
      if (ph.barrier_after) grid_barrier<CT>(P.barrier, bar_target, G);
      if (stamp) stamp[3] = global_ns();
    }

    // ---- greedy id: every CTA folds the per-CTA partials identically (argmax_kernel.cu:49-71
    // semantics: maximum value, lowest index) -------------------------------------------------------
    ArgBest b{0.f, -1};
    for (int c = lane; c < G; c += 32) arg_fold(b, __ldcg(P.arg_val + c), __ldcg(P.arg_idx + c));
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const float ov = __shfl_xor_sync(kFull, b.v, off);
      const int oi = __shfl_xor_sync(kFull, b.i, off);
      arg_fold(b, ov, oi);
    }
    const int next = b.i < 0 ? 0 : b.i;
    if (cta == 0 && tid == 0) {
      if (P.out_tokens != nullptr && step < P.max_steps) P.out_tokens[step] = next;
    }
    token = (P.teacher != nullptr && step + 1 < P.max_steps) ? P.teacher[step + 1] : next;
    if (static_cast<unsigned>(token) >= static_cast<unsigned>(P.vocab_size)) token = 0;
    pos += 1;
    step += 1;
    if (cta == 0 && tid == 0 && tok == P.n_tokens - 1) {
      P.state->token = token;
      P.state->pos = pos;
      P.state->step = step;
      P.state->next = next;
    }
  }
}

}  // namespace mega

// ================================== host side ======================================================
using mega::Params;
using mega::Phase;

namespace {
// PROF: the instantiation kllm_decoder_profile launches (its stamps cost registers in the row loops)
template <bool PROF>
const void* kernel_for(int consumer_warps, bool int8) {
  if (int8) {
    if (consumer_warps == 16) return reinterpret_cast<const void*>(mega::decode_megakernel<16, true, PROF>);
    if (consumer_warps == 14) return reinterpret_cast<const void*>(mega::decode_megakernel<14, true, PROF>);
    if (consumer_warps == 12) return reinterpret_cast<const void*>(mega::decode_megakernel<12, true, PROF>);
    if (consumer_warps == 6) return reinterpret_cast<const void*>(mega::decode_megakernel<6, true, PROF>);
    return reinterpret_cast<const void*>(mega::decode_megakernel<8, true, PROF>);
  }
  if (consumer_warps == 6) return reinterpret_cast<const void*>(mega::decode_megakernel<6, false, PROF>);
  return reinterpret_cast<const void*>(mega::decode_megakernel<8, false, PROF>);
}
}  // namespace

int MegaEngine::init(const MegaModel& m, cudaStream_t stream) {
  model_ = m;
  stream_ = stream;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return KLLM_E_NODEVICE;
  int sms = 0, coop = 0, max_smem = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
  cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  if (!coop) return KLLM_E_UNSUPPORTED;

  const int dim = m.dim, hid = m.hidden_dim, hs = m.head_size, kvd = m.kv_dim;
  const int q_rows = m.head_num * hs;
  const bool int8 = m.group_size > 0;
  const int wb = int8 ? 1 : 4;
  // One CTA per SM, but never more CTAs than the shortest row-parallel phase has rows: the
  // slot-reuse argument of the tagged hand-offs wants every CTA to own rows in every producing
  // phase (a CTA without rows gates nothing and could be overtaken).  Small test shapes only.
  grid_ = std::min(sms, std::min(dim, hid));
  if (grid_ < m.head_num) return KLLM_E_UNSUPPORTED;  // attention: one CTA per (local) query head
  // shapes the ring handles: 16-byte rows, 128-byte aligned kv rows (L1-cached reads stay exact);
  // head_size <= 128: the K-tile producer issues one bulk copy per lane for hs/4 <= 32 chunk columns
  if ((dim & 3) || (hid & 3) || (q_rows & 3) || (hs & 3) || hs > 128) return KLLM_E_UNSUPPORTED;
  if (int8 && ((dim & 15) || (hid & 15) || (q_rows & 15) || (m.group_size & 3))) return KLLM_E_UNSUPPORTED;
  if ((hs * 4) % 16 != 0) return KLLM_E_UNSUPPORTED;
  if (int8) {
    const int dims[3] = {dim, hid, q_rows};
    for (int d : dims)
      if (d % m.group_size != 0 || ((d / m.group_size) * 4) % 16 != 0) return KLLM_E_UNSUPPORTED;
  }
  // consumer warps (+ the ring producer and the L2 prefetcher): fp32 rows 8 x 168 registers; int8 rows 14, so
  // that the CTA is 16 warps = 4 per scheduler with 128 registers each (16 consumers make 18 warps, which caps
  // them at 96 registers and spills).  Measured on B200 (profiles/README.md, passes Q-T): fp32 6 vs 8 warps
  // 1072 = 1072 (TinyLlama), 1218 < 1296 (Qwen2.5-0.5B), 210 < 213 (Llama-2-7B); int8 16 / 14 / 8 warps
  // 394 / 400 / 375 tok/s.
  consumer_warps_ = int8 ? 14 : 8;
  if (const char* e = getenv("KLLM_CONSUMER_WARPS")) {
    const int v = atoi(e);
    if (int8 && (v == 6 || v == 8 || v == 12 || v == 14 || v == 16)) consumer_warps_ = v;  // fast mode: CT >= 192 quantises M <= 16384 in <= 6 rounds
    if (!int8 && (v == 6 || v == 8)) consumer_warps_ = v;
  }
  // int8 arithmetic: "exact" reproduces the reference's fma(x * scale, float(w), acc) per element bit for
  // bit; "fast" (KLLM_INT8_MODE=fast) is the dp4a fixed-point mode (toleranced, ~3.5x fewer instructions)
  // The same switch frees the attention's summation order (flash-decoding, attention_flash_phase).
  // kllm_decoder_desc::numerics picks the mode; KLLM_MODE=exact|fast (KLLM_INT8_MODE: older name) overrides.
  fast_ = m.numerics == 1 ? 1 : 0;
  for (const char* name : {"KLLM_INT8_MODE", "KLLM_MODE"})
    if (const char* e = getenv(name)) fast_ = std::string(e) == "fast" ? 1 : 0;
  int8_fast_ = (int8 && fast_) ? 1 : 0;
  kernel_ = kernel_for<false>(consumer_warps_, int8);
  kernel_prof_ = kernel_for<true>(consumer_warps_, int8);
  threads_ = consumer_warps_ * 32 + 64;

  // Tagged exchange instead of "write x, grid barrier, read x" after o_proj and down_proj:
  // mandatory under tensor parallelism (it IS the all-reduce), optional on one GPU.
  // KLLM_MEGA_TAGGED = 0: grid barriers everywhere (one GPU only); 1: tagged residual exchange;
  // 2 (default): + tagged hand-offs q|k|v -> attention -> Wo and SwiGLU -> W2, which leaves ONE
  // grid barrier per token (after the classifier).
  const int W = m.tp_world > 1 ? m.tp_world : 1;
  if (W != 1 && W != 2 && W != 4 && W != 8) return KLLM_E_UNSUPPORTED;
  tagged_mode_ = 2;
  if (const char* e = getenv("KLLM_MEGA_TAGGED")) tagged_mode_ = std::min(2, std::max(0, atoi(e)));
  if (W > 1 && tagged_mode_ == 0) tagged_mode_ = 1;
  tagged_ = tagged_mode_ >= 1;
  const bool handoffs = tagged_mode_ >= 2;

  // ---- shared memory plan -----------------------------------------------------------------------
  const int max_in = std::max(std::max(dim, hid), q_rows);
  int xbuf = max_in * 4;
  const int attn_ws = 2 * hs * 4;
  xbuf = std::max(xbuf, attn_ws);
  // Stage size: whole rows, so pick it to waste little of the ring on the model's row lengths.
  // fp32: 32 KB (4 rows of dim 2048, 2 of 4096).  int8: 27 KB = 6 rows of dim 4096 (+ scales) or
  // 2 rows of hidden 11008, which leaves six stages next to the 44 KB input vector and the 16 KB
  // residual stream of Llama-2-7B.
  int stage_bytes = int8 ? 27 * 1024 : 32 * 1024;
  if (const char* e = getenv("KLLM_STAGE_BYTES")) stage_bytes = atoi(e);
  stage_bytes = (stage_bytes + 127) & ~127;
  attn_tile_ = std::min(stage_bytes / (hs * 4), consumer_warps_ * 32) & ~31;  // one timestep per consumer thread
  if (attn_tile_ < 32) return KLLM_E_UNSUPPORTED;
  attn_parts_ = 1;
  if (fast_) {  // flash attention: a lane quartet per timestep, warp partials (m, l, o[hs]) in the input buffer
    if (hs & 15) return KLLM_E_UNSUPPORTED;
    xbuf = std::max(xbuf, (2 * hs + consumer_warps_ * (hs + 2)) * 4);
  }
  xbuf = (xbuf + 127) & ~127;
  const int xres = tagged_ ? ((dim * 4 + 127) & ~127) : 0;  // the CTA's copy of the residual stream
  const int budget = max_smem - xbuf - xres - 3584;  // static shared memory (3 KB) + slack
  int stages = budget / stage_bytes;
  if (stages > mega::kMaxStages) stages = mega::kMaxStages;
  if (const char* e = getenv("KLLM_STAGES")) stages = std::min(stages, atoi(e));
  if (stages < 2) return KLLM_E_UNSUPPORTED;
  stage_bytes_ = stage_bytes;
  stages_ = stages;
  // attention split: SP CTAs per query head (power of two, <= 8), each owning head_size / SP output dims
  // (a multiple of 4 floats so that V slice rows stay 16-byte units for the bulk copies)
  if (m.seq_len & 3) return KLLM_E_UNSUPPORTED;
  attn_split_ = 1;
  while (attn_split_ * 2 <= 8 && m.head_num * attn_split_ * 2 <= grid_ && (hs / (attn_split_ * 2)) % 4 == 0 &&
         hs % (attn_split_ * 2) == 0)
    attn_split_ *= 2;
  const int attn_split_max = attn_split_;
  // The split costs one more hand-off per layer (~1.5 us): worth it when a head's K and V are big
  // (head_size 128: 1 MB per head at context 1024), not for head_size 64 (measured, profiles/README.md).
  if (hs < 128) attn_split_ = 1;
  int split_cap = attn_split_max;
  if (fast_) {  // flash: split by timestep, any power of two whose partial triples fit the scores area
    attn_split_ = 1;
    while (attn_split_ * 2 <= 8 && m.head_num * attn_split_ * 2 <= grid_ && attn_split_ * 2 * (hs + 2) <= m.seq_len)
      attn_split_ *= 2;
    split_cap = attn_split_;
  }
  if (const char* e = getenv("KLLM_ATTN_SPLIT")) {
    const int v = atoi(e);
    if (v >= 1 && v <= split_cap && (v & (v - 1)) == 0) attn_split_ = v;
  }
  attn_vsplit_ = fast_ ? 1 : attn_split_;
  attn_tile_v_ = (stage_bytes / ((hs / attn_vsplit_) * 4)) & ~31;
  if (attn_tile_v_ < 32) return KLLM_E_UNSUPPORTED;
  xbuf_bytes_ = xbuf;
  xres_bytes_ = xres;
  smem_bytes_ = static_cast<size_t>(mega::kCtlBytes) + xbuf + xres + static_cast<size_t>(stages) * stage_bytes;

  // ---- phase table ---------------------------------------------------------------------------------
  std::vector<Phase> ph;
  // Rows per consumer task (1, 2 or 4) of a phase.  Measured on B200 (profiles/README.md, passes Q and R):
  // 4 everywhere is best or equal (TinyLlama 1105 vs 1082 "auto" vs 1068 with 2; Llama-2-7B int8 418 / 405 /
  // 407) -- the four rows of a task share every load of the input vector, and that outweighs the better
  // balance of small tasks.  KLLM_TASK_ROWS_RT=1|2|4 forces a size, =auto picks per phase with the cost model
  // below (rounds x (rows + x_cost), tasks never crossing a ring stage).
  int forced_task_rows = 4;
  if (const char* e = getenv("KLLM_TASK_ROWS_RT")) {
    const int v = atoi(e);
    if (v == 1 || v == 2 || v == 4) forced_task_rows = v;
    if (std::string(e) == "auto") forced_task_rows = 0;
  }
  // KLLM_INT8_MMA=1: int8 fast rows in the team form -- mma.sync m16n8k32 s8 for stages of 3-8 rows, dp4a with the
  // columns split over the team for 1-2 long rows.  Correct (the parity suite passes with it) but not faster on
  // B200: Llama-2-7B int8 398 (teams of 4, 12 warps) / 403 (pairs, 14 warps) vs 407 tok/s for the plain dp4a
  // rows (profiles/README.md, passes S and T) -- at one byte per weight the shared-memory reads of the
  // fragments cost what the dp4a arithmetic costs.  Off by default.
  bool int8_mma = false;
  if (const char* e = getenv("KLLM_INT8_MMA")) int8_mma = atoi(e) != 0;
  auto pick_task_rows = [&](Phase& p) {
    const int rpu = p.swiglu ? 2 : 1;
    p.task_rows = 4;
    if (p.chunks_per_row != 1) return;
    if (forced_task_rows) {
      p.task_rows = std::max(forced_task_rows, rpu);
      return;
    }
    const int rows_cta = ((p.units + grid_ - 1) / grid_) * rpu;
    const int rps = std::max(rpu, p.rows_per_stage);
    const double x_cost = int8 ? 0.5 : 1.0;
    double best_cost = 1e30;
    for (int nr : {4, 2, 1}) {
      if (nr < rpu) continue;  // SwiGLU units are row pairs
      int tasks = 0;
      for (int left = rows_cta; left > 0; left -= rps) tasks += (std::min(rps, left) + nr - 1) / nr;
      // tasks never cross a ring stage, so at most stages x (tasks per stage) of them exist at a time
      const int concurrent = std::max(1, std::min(consumer_warps_, stages * ((rps + nr - 1) / nr)));
      const int rounds = (tasks + concurrent - 1) / concurrent;
      const double cost = rounds * (std::min(nr, rps) + x_cost);
      if (cost < best_cost - 1e-9) best_cost = cost, p.task_rows = nr;
    }
  };
  auto plan = [&](Phase& p) -> int {
    const int row_bytes = p.in_dim * wb;
    p.group_size = m.group_size;
    p.group_shift = -1;
    if (int8 && (m.group_size & (m.group_size - 1)) == 0) {
      int s = 0;
      while ((1 << s) < m.group_size) ++s;
      p.group_shift = s;
    }
    p.scale_row_bytes = int8 ? (p.in_dim / m.group_size) * 4 : 0;
    const int rpu = p.swiglu ? 2 : 1;
    // int8 fast mode: stages that hold >= 3 rows go through the tensor cores (accum_w8_mma): <= 8 rows per
    // stage, rows and scale rows staged 16 bytes apart more than their length
    p.mma = 0, p.row_pad = 0, p.team = 0;
    if (int8_fast_ && int8_mma && m.group_size == 64 && p.in_dim % 64 == 0) {
      const int padded = row_bytes + 16 + p.scale_row_bytes + 16;
      int rows = std::min(8, stage_bytes / padded);
      rows -= rows % rpu;
      while (rows >= 3 && ((rows * (row_bytes + 16) + 127) & ~127) + rows * (p.scale_row_bytes + 16) > stage_bytes) rows -= rpu;
      if (rows >= 3) {
        p.mma = 1, p.row_pad = 16, p.team = 1;
        p.rows_per_stage = rows;
        p.chunks_per_row = 1;
        p.chunk_elems = p.in_dim;
        p.scale_off = (rows * (row_bytes + 16) + 127) & ~127;
        pick_task_rows(p);
        return 0;
      }
    }
    const int per_row = row_bytes + p.scale_row_bytes;
    if (per_row * rpu <= stage_bytes) {
      int rows = stage_bytes / per_row;
      rows -= rows % rpu;
      rows = std::min(rows, 32);  // one bulk copy per producer lane
      // int8 fast mode, one or two long rows per stage (hidden_dim columns): a team of warps on dp4a
      if (int8_fast_ && int8_mma && m.group_size == 64 && p.in_dim % 64 == 0 && rows <= 2) p.team = 1;
      p.rows_per_stage = rows;
      p.chunks_per_row = 1;
      p.chunk_elems = p.in_dim;
      p.scale_off = ((rows * row_bytes) + 127) & ~127;
      if (p.scale_off + rows * p.scale_row_bytes > stage_bytes) {
        // shrink until weights + scales fit
        while (rows > rpu && (((rows * row_bytes + 127) & ~127) + rows * p.scale_row_bytes) > stage_bytes)
          rows -= rpu;
        p.rows_per_stage = rows;
        p.scale_off = ((rows * row_bytes) + 127) & ~127;
      }
    } else {
      if (int8 || p.swiglu) return KLLM_E_UNSUPPORTED;
      const int chunk_max = (stage_bytes / 4) & ~511;  // multiple of 128 packs
      p.chunks_per_row = (p.in_dim + chunk_max - 1) / chunk_max;
      int ce = (p.in_dim + p.chunks_per_row - 1) / p.chunks_per_row;
      ce = (ce + 511) & ~511;
      p.chunk_elems = ce;
      p.chunks_per_row = (p.in_dim + ce - 1) / ce;
      p.rows_per_stage = 1;
      p.scale_off = 0;
    }
    pick_task_rows(p);
    return 0;
  };

  unsigned long long *t_q = nullptr, *t_k = nullptr, *t_v = nullptr, *t_attn = nullptr, *t_h = nullptr;
  if (handoffs) {
    const size_t words = static_cast<size_t>(2 * q_rows + 2 * kvd + hid);
    if (cudaMalloc(&d_handoff_, sizeof(unsigned long long) * words) != cudaSuccess)
      return static_cast<int>(cudaErrorMemoryAllocation);
    cudaMemsetAsync(d_handoff_, 0, sizeof(unsigned long long) * words, stream);
    t_q = d_handoff_, t_k = t_q + q_rows, t_v = t_k + kvd, t_attn = t_v + kvd, t_h = t_attn + q_rows;
  }
  {
    const size_t words = static_cast<size_t>(m.head_num) * m.seq_len;
    if (cudaMalloc(&d_scores_, sizeof(unsigned long long) * words) != cudaSuccess)
      return static_cast<int>(cudaErrorMemoryAllocation);
    cudaMemsetAsync(d_scores_, 0, sizeof(unsigned long long) * words, stream);
  }
  int hands = 0;
  if (tagged_ && W == 1) {
    if (cudaMalloc(&d_tagged_, sizeof(unsigned long long) * 2 * dim) != cudaSuccess)
      return static_cast<int>(cudaErrorMemoryAllocation);
    cudaMemsetAsync(d_tagged_, 0, sizeof(unsigned long long) * 2 * dim, stream);
  }
  int exch = 0, bars = 0;
  auto close_phase = [&](Phase& p, bool barrier) {
    p.barrier_after = barrier ? 1 : 0;
    if (barrier) ++bars;
    p.barrier_idx = bars;
  };
  // a phase whose input is the residual stream: tagged -> x_old (shared memory) + partials of the
  // last exchange
  auto input_is_x = [&](Phase& p) {
    if (!tagged_ || exch == 0) {
      p.x = m.x;
      return;
    }
    p.tp_in = 1;
    p.exch = exch - 1;
    p.x = nullptr;
  };
  // a row-parallel matmul whose output is added to the residual stream
  auto output_adds_to_x = [&](Phase& p, bool first_layer) {
    if (tagged_) {
      p.tp_out = 1;
      p.exch_out = exch++;
      p.residual = nullptr;
      p.residual_from_emb = 0;
      close_phase(p, false);
    } else {
      p.residual = m.x;
      p.residual_from_emb = first_layer ? 1 : 0;
      close_phase(p, true);
    }
  };

  const float eps = flavour_eps(m.flavour);
  for (int l = 0; l < m.layer_num; ++l) {
    const size_t layer_off = static_cast<size_t>(l) * m.seq_len * kvd;
    {  // attention_rms + q | k | v (+bias).  k goes to k_raw (rotated later), v into the cache.
      Phase p{};
      p.kind = mega::kPhaseGemv;
      p.in_dim = dim;
      p.n_seg = 3;
      input_is_x(p);
      p.x_from_emb = (l == 0);
      p.norm_w = m.attn_norm[l];
      p.norm_eps = eps;
      p.seg[0] = {m.wq[l], int8 ? m.sq[l] : nullptr, m.bq ? m.bq[l] : nullptr, m.q, 0, q_rows, 0};
      p.seg[1] = {m.wk[l], int8 ? m.sk[l] : nullptr, m.bk ? m.bk[l] : nullptr, m.k_raw, 0, kvd, 0};
      p.seg[2] = {m.wv[l], int8 ? m.sv[l] : nullptr, m.bv ? m.bv[l] : nullptr,
                  m.value_cache + layer_off, 0, kvd, 1};
      p.units = q_rows + 2 * kvd;
      if (int rc = plan(p)) return rc;
      if (handoffs) {  // q, raw k: tagged only; v: cache row (for later tokens) + tagged (for this one)
        p.seg[0].out = nullptr, p.seg[0].tag_out = t_q;
        p.seg[1].out = nullptr, p.seg[1].tag_out = t_k;
        p.seg[2].tag_out = t_v;
        p.hand_out = hands;
      }
      close_phase(p, !handoffs);
      ph.push_back(p);
    }
    if (fast_) {  // flash-decoding: attn_split_ CTAs per head by timestep, one phase
      Phase p{};
      p.kind = mega::kPhaseAttnFlash;
      p.layer = l;
      if (handoffs) {
        p.tq = t_q, p.tk = t_k, p.tv = t_v, p.ta = t_attn;
        p.hand_in = hands++;
        p.hand_out = hands;
      } else {
        p.hand_out = hands++;  // the partial (m, l, o) triples are tagged words in every mode
      }
      close_phase(p, !handoffs);
      ph.push_back(p);
    } else if (attn_split_ == 1) {  // one CTA per head, one phase
      Phase p{};
      p.kind = mega::kPhaseAttnFused;
      p.layer = l;
      if (handoffs) {
        p.tq = t_q, p.tk = t_k, p.tv = t_v, p.ta = t_attn;
        p.hand_in = hands++;
        p.hand_out = hands;
      }
      close_phase(p, !handoffs);
      ph.push_back(p);
    } else {
      int qkv_hand = 0;
      {  // attention, scores: CTA (head, s) scores the K tiles s, s + SP, ... and publishes them tagged
        Phase p{};
        p.kind = mega::kPhaseAttention;
        p.layer = l;
        if (handoffs) {
          p.tq = t_q, p.tk = t_k, p.tv = t_v;
          p.hand_in = hands++;
        }
        qkv_hand = p.hand_in;
        p.hand_out = hands;  // the scores (always tagged words, also in the barrier modes)
        close_phase(p, !handoffs);
        ph.push_back(p);
      }
      {  // attention, softmax + P.V: CTA (head, s) owns output dims [s dv, (s + 1) dv)
        Phase p{};
        p.kind = mega::kPhaseAttnPV;
        p.layer = l;
        p.hand_in = hands++;
        if (handoffs) {
          p.tv = t_v, p.ta = t_attn;
          p.hand_aux = qkv_hand;
          p.hand_out = hands;
        }
        close_phase(p, !handoffs);
        ph.push_back(p);
      }
    }
    {  // wo + residual (llama3.cpp:672-684)
      Phase p{};
      p.kind = mega::kPhaseGemv;
      p.in_dim = q_rows;
      p.n_seg = 1;
      p.x = m.attn_out;
      p.seg[0] = {m.wo[l], int8 ? m.so[l] : nullptr, nullptr, m.x, 0, dim, 0};
      p.units = dim;
      if (handoffs) {
        p.tag_in = t_attn;
        p.hand_in = hands++;
        p.x = nullptr;
      }
      if (int rc = plan(p)) return rc;
      output_adds_to_x(p, l == 0);
      ph.push_back(p);
    }
    {  // ffn rmsnorm + w1 | w3 -> swiglu (llama3.cpp:686-708)
      Phase p{};
      p.kind = mega::kPhaseGemv;
      p.in_dim = dim;
      p.n_seg = 2;
      p.swiglu = 1;
      input_is_x(p);
      p.norm_w = m.ffn_norm[l];
      p.norm_eps = eps;
      p.seg[0] = {m.w1[l], int8 ? m.s1[l] : nullptr, nullptr, m.h, 0, hid, 0};
      p.seg[1] = {m.w3[l], int8 ? m.s3[l] : nullptr, nullptr, nullptr, 0, hid, 0};
      p.units = hid;
      if (int rc = plan(p)) return rc;
      if (handoffs) {
        p.seg[0].out = nullptr, p.seg[0].tag_out = t_h;
        p.hand_out = hands;
      }
      close_phase(p, !handoffs);
      ph.push_back(p);
    }
    {  // w2 + residual (llama3.cpp:711-719)
      Phase p{};
      p.kind = mega::kPhaseGemv;
      p.in_dim = hid;
      p.n_seg = 1;
      p.x = m.h;
      p.seg[0] = {m.w2[l], int8 ? m.s2[l] : nullptr, nullptr, m.x, 0, dim, 0};
      p.units = dim;
      if (handoffs) {
        p.tag_in = t_h;
        p.hand_in = hands++;
        p.x = nullptr;
      }
      if (int rc = plan(p)) return rc;
      output_adds_to_x(p, false);
      ph.push_back(p);
    }
  }
  {  // final rmsnorm + classifier (+ argmax partials)
    Phase p{};
    p.kind = mega::kPhaseGemv;
    p.in_dim = dim;
    p.n_seg = 1;
    input_is_x(p);
    p.norm_w = m.final_norm;
    p.norm_eps = eps;
    p.cls = 1;
    // Tensor parallel: shard the classifier by vocabulary when the exchange area can carry a rank's
    // rows (kllm_comm_create(max_count >= vocab / world)); every rank still holds the whole matrix and
    // reads only its rows.  KLLM_TP_SHARD_CLS=0 keeps it replicated.
    const char* shard_env = getenv("KLLM_TP_SHARD_CLS");
    const bool shard = W > 1 && m.vocab_size % W == 0 && m.tp_stride >= m.vocab_size / W &&
                       !(shard_env && atoi(shard_env) == 0);
    cls_rows_ = shard ? m.vocab_size / W : m.vocab_size;
    n_cls_phases_ = shard ? 2 : 1;
    if (shard) {
      const size_t row0 = static_cast<size_t>(m.tp_rank) * cls_rows_;
      p.seg[0] = {static_cast<const unsigned char*>(m.wcls) + row0 * dim * wb,
                  int8 ? m.scls + row0 * (dim / m.group_size) : nullptr, nullptr, nullptr, 0, cls_rows_, 0};
      p.units = cls_rows_;
      if (int rc = plan(p)) return rc;
      p.tp_out = 1;  // rows go to every rank's exchange area as tagged words
      p.exch_out = exch++;
      close_phase(p, false);
      ph.push_back(p);
      Phase g{};
      g.kind = mega::kPhaseGather;
      g.cls = 1;
      g.argmax = 1;
      g.units = m.vocab_size;
      g.in_dim = cls_rows_;
      g.exch = p.exch_out;
      g.seg[0].out = m.logits;
      close_phase(g, true);
      ph.push_back(g);
    } else {
      p.seg[0] = {m.wcls, int8 ? m.scls : nullptr, nullptr, m.logits, 0, m.vocab_size, 0};
      p.units = m.vocab_size;
      p.argmax = 1;
      if (int rc = plan(p)) return rc;
      close_phase(p, true);
      ph.push_back(p);
    }
  }
  n_phases_ = static_cast<int>(ph.size());
  n_barriers_per_token_ = bars;
  exch_per_token_ = exch;
  hands_per_token_ = hands;
  // The producer streams K/V rows written by the PREVIOUS token once the grid barrier that closed
  // that token's attention phase is passed; without such a barrier, the one that closed the token.
  for (Phase& p : ph)
    if (p.kind != mega::kPhaseGemv && !p.barrier_after) p.barrier_idx = bars;

  if (cudaMalloc(&d_phases_, sizeof(Phase) * ph.size()) != cudaSuccess) return static_cast<int>(cudaErrorMemoryAllocation);
  cudaMemcpyAsync(d_phases_, ph.data(), sizeof(Phase) * ph.size(), cudaMemcpyHostToDevice, stream);
  if (cudaMalloc(&d_barrier_, 128) != cudaSuccess) return static_cast<int>(cudaErrorMemoryAllocation);
  cudaMemsetAsync(d_barrier_, 0, 128, stream);
  if (cudaMalloc(&d_arg_val_, sizeof(float) * grid_) != cudaSuccess ||
      cudaMalloc(&d_arg_idx_, sizeof(int) * grid_) != cudaSuccess)
    return static_cast<int>(cudaErrorMemoryAllocation);
  cudaStreamSynchronize(stream);  // ph (host vector) must outlive the async copy

  cudaError_t e = cudaFuncSetAttribute(kernel_, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(smem_bytes_));
  if (e != cudaSuccess) return static_cast<int>(e);
  e = cudaFuncSetAttribute(kernel_prof_, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem_bytes_));
  if (e != cudaSuccess) return static_cast<int>(e);
  int occ = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel_, threads_, smem_bytes_);
  if (e != cudaSuccess) return static_cast<int>(e);
  if (occ < 1) return KLLM_E_UNSUPPORTED;
  barrier_base_ = 0;
  ready_ = true;
  return 0;
}

void MegaEngine::destroy() {
  if (d_phases_) cudaFree(d_phases_);
  if (d_barrier_) cudaFree(d_barrier_);
  if (d_arg_val_) cudaFree(d_arg_val_);
  if (d_arg_idx_) cudaFree(d_arg_idx_);
  if (d_tagged_) cudaFree(d_tagged_);
  if (d_handoff_) cudaFree(d_handoff_);
  if (d_scores_) cudaFree(d_scores_);
  d_scores_ = nullptr;
  d_handoff_ = nullptr;
  d_tagged_ = nullptr;
  d_phases_ = nullptr;
  d_barrier_ = nullptr;
  d_arg_val_ = nullptr;
  d_arg_idx_ = nullptr;
  ready_ = false;
}

int MegaEngine::run(int n_tokens, const int32_t* teacher_dev, unsigned long long* prof_dev,
                    int prof_token, int skip_cls_tokens) {
  if (!ready_) return KLLM_E_STATE;
  Params P{};
  const MegaModel& m = model_;
  P.phases = static_cast<const Phase*>(d_phases_);
  P.n_phases = n_phases_;
  P.n_tokens = n_tokens;
  P.skip_cls_tokens = skip_cls_tokens;
  P.n_cls_phases = n_cls_phases_;
  P.int8_fast = int8_fast_;
  P.num_stages = stages_;
  P.stage_bytes = stage_bytes_;
  P.xbuf_bytes = xbuf_bytes_;
  P.xres_bytes = xres_bytes_;
  P.attn_tile = attn_tile_;
  P.attn_tile_v = attn_tile_v_;
  P.attn_split = attn_split_;
  P.attn_vsplit = attn_vsplit_;
  P.attn_parts = attn_parts_;
  P.scores = d_scores_;
  // 256 KB per SM = 38 MB of weights in flight towards L2 chip-wide (measured with 32 KB stages: 6-12 stages
  // best, >= 24 thrashes L2); in stages, so that a smaller stage size keeps the same byte distance
  P.pf_stages = std::max(4, (256 * 1024) / std::max(1, stage_bytes_));
  if (const char* e = getenv("KLLM_PREFETCH_STAGES")) P.pf_stages = std::max(0, atoi(e));
  P.group_size = m.group_size;
  P.dim = m.dim;
  P.vocab_size = m.vocab_size;
  P.head_num = m.head_num;
  P.head_size = m.head_size;
  P.kv_dim = m.kv_dim;
  P.kv_mul = m.kv_mul;
  P.seq_len = m.seq_len;
  P.flavour = m.flavour;
  P.tok_emb = m.tok_emb;
  P.q = m.q;
  P.k_raw = m.k_raw;
  P.attn_out = m.attn_out;
  P.score = m.score;
  P.key_cache = m.key_cache;
  P.value_cache = m.value_cache;
  P.sin_cache = m.sin_cache;
  P.cos_cache = m.cos_cache;
  P.state = static_cast<mega::State*>(m.state);
  P.out_tokens = m.out_tokens;
  P.teacher = teacher_dev;
  P.max_steps = m.seq_len;
  P.barrier = static_cast<unsigned*>(d_barrier_);
  P.barrier_base = barrier_base_;
  P.bars_per_token = n_barriers_per_token_;
  P.tp_world = m.tp_world > 1 ? m.tp_world : 1;
  P.tp_rank = m.tp_world > 1 ? m.tp_rank : 0;
  P.tp_stride = m.tp_world > 1 ? m.tp_stride : m.dim;
  for (int r = 0; r < 8; ++r) P.tp_data[r] = m.tp_world > 1 ? m.tp_data[r] : nullptr;
  if (m.tp_world <= 1) P.tp_data[0] = d_tagged_;
  P.exch_per_token = exch_per_token_;
  P.tp_seq_base = tp_seq_base_;
  P.hand_base = hand_base_;
  P.hands_per_token = hands_per_token_;
  P.arg_val = static_cast<float*>(d_arg_val_);
  P.arg_idx = static_cast<int*>(d_arg_idx_);
  P.prof = prof_dev;
  P.prof_token = prof_token;
  void* args[] = {&P};
  cudaError_t e = cudaLaunchCooperativeKernel(const_cast<void*>(prof_dev != nullptr ? kernel_prof_ : kernel_), dim3(grid_), dim3(threads_), args,
                                              smem_bytes_, stream_);
  if (e != cudaSuccess) return static_cast<int>(e);
  tp_seq_base_ += static_cast<unsigned>(n_tokens) * static_cast<unsigned>(exch_per_token_);
  hand_base_ += static_cast<unsigned>(n_tokens) * static_cast<unsigned>(hands_per_token_);
  barrier_base_ += static_cast<unsigned>(n_tokens) * static_cast<unsigned>(n_barriers_per_token_) *
                   static_cast<unsigned>(grid_);
  count_launch();
  return 0;
}

}  // namespace kllm
