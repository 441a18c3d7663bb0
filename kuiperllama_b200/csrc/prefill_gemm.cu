// Batched GEMM for prompt prefill on the 5th-generation tensor cores (sm_100a):
//     out[T, N] = x[T, K] . w[N, K]^T        fp32 storage, TF32 multiply, fp32 accumulate in TMEM
//
// The reference feeds a prompt through one full single-token forward per position (demo/main.cpp:
// 18-23, llama3.cpp:147-167) -- T GEMVs that stream every weight T times.  With the T prompt rows
// as the N dimension of a tcgen05.mma the weights are streamed once per 256 tokens.
//
// This is an explicitly TOLERANCED kernel: TF32 keeps 10 mantissa bits of each operand, so results
// agree with the fp32 GEMV path to ~1e-3 relative, not bit for bit (tests/test_prefill_gpu.py states
// the bound).  The bit-exact decode path never calls it.
//
// Structure (one CTA per 128 weight rows x one block of BN tokens, 6 warps):
//   warp 0   TMA producer: cp.async.bulk.tensor 2-D tiles of w [128 x 32 fp32] and x [BN x 32 fp32],
//            128-byte swizzle, into a 4-stage shared-memory ring (SASS: UTMALDG)
//   warp 1   MMA issuer: one thread, 4 x tcgen05.mma.kind::tf32 (M 128, N BN, K 8) per stage, D in
//            TMEM; tcgen05.commit frees the stage / signals the epilogue (SASS: UTCHMMA / UTCBAR)
//   warps 2-5 epilogue: tcgen05.ld 32 lanes x 32 columns per warp (SASS: LDTM), transposed store
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdint>

#include "../../include/kllm_b200.h"
#include "kllm_device.cuh"
#include "kllm_host.h"

namespace kllm {
namespace tc {

constexpr int BM = 128;     // weight rows per CTA = MMA M
constexpr int BK = 32;      // fp32 elements per K block = 128 bytes = one swizzle-128B row
constexpr int UMMA_K = 8;   // tf32: 32 bytes of K per tcgen05.mma
constexpr int STAGES = 4;
constexpr int A_BYTES = BM * BK * 4;  // 16 KB
constexpr int THREADS = 192;

__device__ __forceinline__ uint32_t smem_addr(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n .reg .pred p;\n WAIT_%=:\n"
      " mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      " @p bra DONE_%=;\n bra WAIT_%=;\n DONE_%=:\n}" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
// Shared-memory matrix descriptor of a K-major tile with 128-byte swizzle (cute::UMMA::SmemDescriptor,
// cutlass include/cute/arch/mma_sm100_desc.hpp): start address >> 4 in bits [0,14), leading byte
// offset (unused with swizzle; 1) in [16,30), stride byte offset = 8 rows x 128 B = 1024 B >> 4 in
// [32,46), descriptor version 1 in [46,48), layout type SWIZZLE_128B = 2 in [61,64).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
  return static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): D = F32 (1 << 4), A = B = TF32 (2 << 7, 2 << 10),
// both K-major (bits 15, 16 clear), N >> 3 in [17,23), M >> 4 in [24,29).
__device__ __forceinline__ uint32_t umma_idesc_tf32(int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(BM >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n"
      " tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

template <int BN>
__global__ void __launch_bounds__(THREADS, 1)
gemm_tf32_kernel(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_x,
                 float* __restrict__ out, int T, int N, int K) {
  constexpr int B_BYTES = BN * BK * 4;
  constexpr uint32_t TMEM_COLS = BN < 32 ? 32 : BN;  // power of two >= 32
  extern __shared__ uint8_t raw_smem[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw_smem) + 1023) & ~uintptr_t(1023));
  uint8_t* a_tiles = base;
  uint8_t* b_tiles = base + STAGES * A_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(b_tiles + STAGES * B_BYTES);
  uint64_t* full = bars;
  uint64_t* empty = bars + STAGES;
  uint64_t* tmem_full = bars + 2 * STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = blockIdx.x * BM;  // first weight row (output feature) of this CTA
  const int t0 = blockIdx.y * BN;  // first token
  const int kblocks = (K + BK - 1) / BK;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(smem_addr(&full[s]), 1);
      mbar_init(smem_addr(&empty[s]), 1);
    }
    mbar_init(smem_addr(tmem_full), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {  // one warp allocates the accumulator's TMEM columns and later frees them
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_addr(tmem_slot)),
                 "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_d = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {  // ---- TMA producer ----
      for (int kb = 0; kb < kblocks; ++kb) {
        const int s = kb % STAGES;
        const uint32_t ph = (kb / STAGES) & 1;
        mbar_wait(smem_addr(&empty[s]), ph ^ 1u);
        const uint32_t bar = smem_addr(&full[s]);
        mbar_expect_tx(bar, A_BYTES + B_BYTES);  // out-of-range rows / columns are zero-filled and still counted
        tma_load_2d(smem_addr(a_tiles + s * A_BYTES), &map_w, bar, kb * BK, n0);
        tma_load_2d(smem_addr(b_tiles + s * B_BYTES), &map_x, bar, kb * BK, t0);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {  // ---- MMA issuer ----
      const uint32_t idesc = umma_idesc_tf32(BN);
      for (int kb = 0; kb < kblocks; ++kb) {
        const int s = kb % STAGES;
        const uint32_t ph = (kb / STAGES) & 1;
        mbar_wait(smem_addr(&full[s]), ph);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t a_addr = smem_addr(a_tiles + s * A_BYTES);
        const uint32_t b_addr = smem_addr(b_tiles + s * B_BYTES);
#pragma unroll
        for (int k = 0; k < BK / UMMA_K; ++k)  // 32 bytes of K per instruction: step inside the swizzle atom
          umma_tf32(tmem_d, umma_desc_sw128(a_addr + k * UMMA_K * 4), umma_desc_sw128(b_addr + k * UMMA_K * 4), idesc,
                    (kb > 0 || k > 0) ? 1u : 0u);
        umma_commit(smem_addr(&empty[s]));  // the stage may be refilled once these MMAs have read it
      }
      umma_commit(smem_addr(tmem_full));  // accumulator complete
    }
  } else {
    // ---- epilogue: TMEM lane = weight row, column = token; a warp may touch lanes 32 (warp % 4) .. +31 ----
    const int quarter = warp & 3;
    mbar_wait(smem_addr(tmem_full), 0u);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const int row = n0 + quarter * 32 + lane;
#pragma unroll 1
    for (int c = 0; c < BN; c += 32) {
      uint32_t r[32];
      const uint32_t taddr = tmem_d + (static_cast<uint32_t>(quarter * 32) << 16) + static_cast<uint32_t>(c);
      asm volatile(
          "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
          "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
          "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
          : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
            "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
            "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
            "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
          : "r"(taddr)
          : "memory");
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      if (row < N) {
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const int t = t0 + c + j;
          if (t < T) out[static_cast<size_t>(t) * N + row] = __uint_as_float(r[j]);  // lanes = consecutive rows: coalesced
        }
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(TMEM_COLS) : "memory");
  }
}

// ---- int8 weights x fixed-point activations on tcgen05.mma.kind::i8 -----------------------------------------
//     out[T, N] = x[T, K] . (s (.) w)[N, K]^T        w int8, s fp32 per (row, 64-group), x fp32
// The activations take the fast decode mode's fixed-point form (kllm_device.cuh, w8_digits4): per token and
// 64-group, x_i ~= step * (65536 a2_i + 256 a1_i + a0_i) with int8 digits.  For weight row r and group g
//     sum_i w_ri x_i = step * (65536 D2 + 256 D1 + D0),   D_k = sum_i w_ri a_k,i   (exact in int32, |D| <= 2^20)
// so one MMA with the three digit planes stacked as B gives all three D's of a group at once:
//   A = 128 weight rows x 128 bytes of K (two groups), B = 3 planes x 64 tokens = 192 rows x 128 bytes,
//   D = s32 [128 x 192] in TMEM, two K = 32 MMAs per group, a FRESH accumulator per group.
// The accumulators are double-buffered in TMEM (columns 0.. and 256.., full / empty mbarriers like the ring),
// so the MMAs of group g + 1 run while the epilogue folds group g into fp32 running sums on CUDA cores:
//     acc[t] += (s[r,g] * step[t,g]) * (65536 D2 + 256 D1 + D0)          (accum_w8_dp4a's arithmetic)
// Only x is rounded (to 2^-23 of its group maximum); weights and scales enter exactly.
//   warp 0     TMA producer: w box [128 x 128 B], planes box [3 x 64 x 128 B], 128-byte swizzle, 4 stages
//   warp 1     MMA issuer (one thread) + TMEM allocation
//   warps 2-9  epilogue: thread = TMEM lane = weight row; two warps per TMEM lane quadrant, each with the fp32
//              running sums of 32 of the 64 tokens in registers (one warp per quadrant cannot hide the
//              latency of the TMEM reads and step loads of a group behind the next group's MMAs)
constexpr int W8_BN = 64;                 // tokens per CTA
constexpr int W8_N = 3 * W8_BN;           // MMA N: the three digit planes of the token tile
constexpr int W8_BK = 128;                // int8 per K block = one swizzle row = two 64-groups
constexpr int W8_UMMA_K = 32;             // kind::i8: 32 bytes of K per tcgen05.mma
constexpr int W8_A_BYTES = BM * W8_BK;    // 16 KB
constexpr int W8_B_BYTES = W8_N * W8_BK;  // 24 KB
constexpr int W8_EPI_WARPS = 8;
constexpr int W8_EPI_TOK = W8_BN * 4 / W8_EPI_WARPS;  // tokens per epilogue thread
constexpr int W8_THREADS = 64 + 32 * W8_EPI_WARPS;
constexpr uint32_t W8_TMEM_COLS = 512;    // accumulator buffers at columns 0 and 256 (192 used each)
constexpr size_t W8_SMEM = 1024 + static_cast<size_t>(STAGES) * (W8_A_BYTES + W8_B_BYTES) + 256;

__device__ __forceinline__ void prefetch_l1(const void* p) {
  asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): D = S32 (2 << 4), A = B = signed 8-bit (1 << 7, 1 << 10),
// both K-major, N >> 3 in [17,23), M >> 4 in [24,29).
__device__ __forceinline__ uint32_t umma_idesc_i8(int n) {
  return (2u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(BM >> 4) << 24);
}
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n"
      " tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// exact int32 -> fp32 for |d| < 2^22 (megakernel.cu small_int_to_float): 1.5 * 2^23 + d is exact
__device__ __forceinline__ float w8_small_int_to_float(uint32_t d) {
  return __fsub_rn(__uint_as_float(0x4B400000u + d), 12582912.0f);
}

// x [T, K] fp32 -> digit planes [3][T][K] int8 and steps [K / 64][t_pad] fp32 (t_pad = T rounded up to 64;
// the pad tokens get step 0).  grid = t_pad, one thread per 16 elements, four lanes per group.
__global__ void __launch_bounds__(256)
quantize_w8_rows_kernel(const float* __restrict__ x, uint8_t* __restrict__ planes, float* __restrict__ steps,
                        int T, int K, int t_pad) {
  const int t = blockIdx.x, quarters = K >> 4;
  const size_t plane = static_cast<size_t>(T) * K;
  for (int base = 0; base < quarters; base += blockDim.x) {  // blockDim % 32 == 0: groups never straddle a warp
    const int qg = base + threadIdx.x;
    const bool on = t < T && qg < quarters;
    float4 v[4];
    float gmax = 0.f;
    const float4* g4 = reinterpret_cast<const float4*>(x + static_cast<size_t>(on ? t : 0) * K) + (on ? qg : 0) * 4;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      v[j] = on ? g4[j] : make_float4(0.f, 0.f, 0.f, 0.f);
      gmax = fmaxf(gmax, fmaxf(fmaxf(fabsf(v[j].x), fabsf(v[j].y)), fmaxf(fabsf(v[j].z), fabsf(v[j].w))));
    }
    gmax = fmaxf(gmax, __shfl_xor_sync(kFull, gmax, 1));
    gmax = fmaxf(gmax, __shfl_xor_sync(kFull, gmax, 2));
    const float inv = w8_group_inv(gmax);
    if (on) {
      uint32_t p[3][4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float e[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
        w8_digits4(e, inv, p[0][j], p[1][j], p[2][j]);
      }
      uint8_t* o = planes + static_cast<size_t>(t) * K + qg * 16;
#pragma unroll
      for (int k = 0; k < 3; ++k)
        *reinterpret_cast<uint4*>(o + k * plane) = make_uint4(p[k][0], p[k][1], p[k][2], p[k][3]);
    }
    if (qg < quarters && (qg & 3) == 0) steps[static_cast<size_t>(qg >> 2) * t_pad + t] = on ? w8_group_step(gmax) : 0.f;
  }
}

__global__ void __launch_bounds__(W8_THREADS, 1)
gemm_w8_kernel(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_p,
               const float* __restrict__ scales, const float* __restrict__ steps, float* __restrict__ out, int T, int N,
               int K, int t_pad) {
  extern __shared__ uint8_t raw_smem[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw_smem) + 1023) & ~uintptr_t(1023));
  uint8_t* a_tiles = base;
  uint8_t* b_tiles = base + STAGES * W8_A_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(b_tiles + STAGES * W8_B_BYTES);
  uint64_t* full = bars;
  uint64_t* empty = bars + STAGES;
  uint64_t* tmem_full = bars + 2 * STAGES;       // [2] MMA -> epilogue: accumulator buffer holds a finished group
  uint64_t* tmem_empty = bars + 2 * STAGES + 2;  // [2] epilogue -> MMA: accumulator buffer read out
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int t0 = blockIdx.x * W8_BN;  // token tiles vary fastest: the CTAs sharing a weight tile run together
  const int n0 = blockIdx.y * BM;
  const int groups = K >> 6, kblocks = (K + W8_BK - 1) / W8_BK;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(smem_addr(&full[s]), 1);
      mbar_init(smem_addr(&empty[s]), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_addr(&tmem_full[b]), 1);
      mbar_init(smem_addr(&tmem_empty[b]), W8_EPI_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_addr(tmem_slot)),
                 "r"(W8_TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_d = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {  // ---- TMA producer ----
      for (int kb = 0; kb < kblocks; ++kb) {
        const int s = kb % STAGES;
        const uint32_t ph = (kb / STAGES) & 1;
        mbar_wait(smem_addr(&empty[s]), ph ^ 1u);
        const uint32_t bar = smem_addr(&full[s]);
        mbar_expect_tx(bar, W8_A_BYTES + W8_B_BYTES);  // zero-filled out-of-range bytes are counted too
        tma_load_2d(smem_addr(a_tiles + s * W8_A_BYTES), &map_w, bar, kb * W8_BK, n0);
        tma_load_3d(smem_addr(b_tiles + s * W8_B_BYTES), &map_p, bar, kb * W8_BK, t0, 0);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {  // ---- MMA issuer ----
      const uint32_t idesc = umma_idesc_i8(W8_N);
      for (int g = 0; g < groups; ++g) {
        const int kb = g >> 1, half = g & 1, s = kb % STAGES, buf = g & 1;
        if (half == 0) {
          mbar_wait(smem_addr(&full[s]), (kb / STAGES) & 1);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
        mbar_wait(smem_addr(&tmem_empty[buf]), ((g >> 1) & 1) ^ 1u);  // the epilogue has read this buffer's last use
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t a_addr = smem_addr(a_tiles + s * W8_A_BYTES) + half * 64;
        const uint32_t b_addr = smem_addr(b_tiles + s * W8_B_BYTES) + half * 64;
        const uint32_t d = tmem_d + static_cast<uint32_t>(buf * 256);
#pragma unroll
        for (int k = 0; k < 64 / W8_UMMA_K; ++k)  // 32 bytes of K per instruction: step inside the swizzle atom
          umma_i8(d, umma_desc_sw128(a_addr + k * W8_UMMA_K), umma_desc_sw128(b_addr + k * W8_UMMA_K), idesc,
                  k > 0 ? 1u : 0u);  // a fresh accumulator per group
        // free the stage once both of its groups are issued -- only if the producer will refill it, so no
        // arrive is left in flight when the CTA exits
        if ((half == 1 || g == groups - 1) && kb + STAGES < kblocks) umma_commit(smem_addr(&empty[s]));
        umma_commit(smem_addr(&tmem_full[buf]));
      }
    }
  } else {
    // ---- epilogue: TMEM lane = weight row; columns p * 64 + t = digit plane p of token t0 + t ----
    const int quarter = warp & 3;  // a warp may touch TMEM lanes 32 (warp % 4) .. +31
    const int tok0 = ((warp - 2) >> 2) * W8_EPI_TOK;  // this warp's tokens: t0 + tok0 .. + W8_EPI_TOK - 1
    const int row = n0 + quarter * 32 + lane;
    const bool row_ok = row < N;
    const float* srow = scales + static_cast<size_t>(row_ok ? row : 0) * groups;
    const uint32_t lane_base = tmem_d + (static_cast<uint32_t>(quarter * 32) << 16);
    float acc[W8_EPI_TOK];
#pragma unroll
    for (int t = 0; t < W8_EPI_TOK; ++t) acc[t] = 0.f;
    const float* st_base = steps + t0 + tok0;  // 128-byte aligned: t_pad, t0 multiples of 64, tok0 of 32
    prefetch_l1(st_base);
#pragma unroll 1
    for (int g = 0; g < groups; ++g) {
      const int buf = g & 1;
      const float ws = row_ok ? __ldg(srow + g) : 0.f;
      const float4* st = reinterpret_cast<const float4*>(st_base + static_cast<size_t>(g) * t_pad);
      if (g + 1 < groups) {  // the next group's steps and scale, so its loads do not wait on L2
        prefetch_l1(st_base + static_cast<size_t>(g + 1) * t_pad);
        prefetch_l1(srow + g + 1);
      }
      mbar_wait(smem_addr(&tmem_full[buf]), (g >> 1) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t cols = lane_base + static_cast<uint32_t>(buf * 256 + tok0);
#pragma unroll
      for (int c = 0; c < W8_EPI_TOK; c += 16) {
        uint32_t d0[16], d1[16], d2[16];
        tmem_ld16(cols + c, d0);
        tmem_ld16(cols + W8_BN + c, d1);
        tmem_ld16(cols + 2 * W8_BN + c, d2);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4) {
          const float4 xs4 = __ldg(st + (c >> 2) + j4);  // same address in every lane: one broadcast
          const float xs[4] = {xs4.x, xs4.y, xs4.z, xs4.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int j = j4 * 4 + e;
            const float f = __fmaf_rn(w8_small_int_to_float(d2[j]), 65536.0f,
                                      __fmaf_rn(w8_small_int_to_float(d1[j]), 256.0f, w8_small_int_to_float(d0[j])));
            acc[c + j] = __fmaf_rn(f, __fmul_rn(xs[e], ws), acc[c + j]);
          }
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_addr(&tmem_empty[buf]));
    }
    if (row_ok) {
#pragma unroll
      for (int t = 0; t < W8_EPI_TOK; ++t)
        if (t0 + tok0 + t < T) out[static_cast<size_t>(t0 + tok0 + t) * N + row] = acc[t];  // lanes = consecutive rows
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(W8_TMEM_COLS) : "memory");
  }
}

// cuTensorMapEncodeTiled comes from the driver (libcuda); it is looked up at run time so that the
// library links and loads on a machine without a driver (the build box).
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}
// Tensor map with 128-byte swizzle over a `rank`-dimensional tensor (dims innermost first, strides in
// bytes for dims 1..rank-1); out-of-range elements of a box are zero-filled.
static int make_map_sw128(CUtensorMap* map, CUtensorMapDataType dtype, const void* ptr, int rank,
                          const cuuint64_t* dims, const cuuint64_t* strides, const cuuint32_t* box) {
  EncodeTiledFn fn = encode_tiled();
  if (fn == nullptr) return KLLM_E_NODEVICE;
  const cuuint32_t estr[3] = {1, 1, 1};
  const CUresult r = fn(map, dtype, static_cast<cuuint32_t>(rank), const_cast<void*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : KLLM_E_INVALID;
}
// 2-D fp32 tensor [rows, cols] (row-major, cols contiguous), box [box_rows x 32 columns], 128-byte swizzle
static int make_map(CUtensorMap* map, const float* ptr, int rows, int cols, int box_rows) {
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(cols) * 4};
  const cuuint32_t box[2] = {static_cast<cuuint32_t>(BK), static_cast<cuuint32_t>(box_rows)};
  return make_map_sw128(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, ptr, 2, dims, strides, box);
}

template <int BN>
static int launch(const float* x, const float* w, float* out, int T, int K, int N, cudaStream_t stream) {
  CUtensorMap map_w, map_x;
  if (int rc = make_map(&map_w, w, N, K, BM)) return rc;
  if (int rc = make_map(&map_x, x, T, K, BN)) return rc;
  const size_t smem = 1024 + static_cast<size_t>(STAGES) * (A_BYTES + BN * BK * 4) + 256;
  static bool configured = false;
  if (!configured) {
    const cudaError_t e = cudaFuncSetAttribute(gemm_tf32_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               static_cast<int>(smem));
    if (e != cudaSuccess) return static_cast<int>(e);
    configured = true;
  }
  const dim3 grid((N + BM - 1) / BM, (T + BN - 1) / BN);
  gemm_tf32_kernel<BN><<<grid, THREADS, smem, stream>>>(map_w, map_x, out, T, N, K);
  count_launch();
  return static_cast<int>(cudaGetLastError());
}

static int launch_w8(const float* x, const int8_t* w, const float* scales, float* out, void* workspace, int T, int K,
                     int N, cudaStream_t stream) {
  const int t_pad = (T + W8_BN - 1) / W8_BN * W8_BN;
  uint8_t* planes = static_cast<uint8_t*>(workspace);
  float* steps = reinterpret_cast<float*>(planes + 3 * static_cast<size_t>(T) * K);  // 3 T K % 64 == 0: aligned
  CUtensorMap map_w, map_p;
  {
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(K), static_cast<cuuint64_t>(N)};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(K)};
    const cuuint32_t box[2] = {static_cast<cuuint32_t>(W8_BK), static_cast<cuuint32_t>(BM)};
    if (int rc = make_map_sw128(&map_w, CU_TENSOR_MAP_DATA_TYPE_UINT8, w, 2, dims, strides, box)) return rc;
  }
  {
    const cuuint64_t dims[3] = {static_cast<cuuint64_t>(K), static_cast<cuuint64_t>(T), 3};
    const cuuint64_t strides[2] = {static_cast<cuuint64_t>(K), static_cast<cuuint64_t>(T) * K};
    const cuuint32_t box[3] = {static_cast<cuuint32_t>(W8_BK), static_cast<cuuint32_t>(W8_BN), 3};
    if (int rc = make_map_sw128(&map_p, CU_TENSOR_MAP_DATA_TYPE_UINT8, planes, 3, dims, strides, box)) return rc;
  }
  static bool configured = false;
  if (!configured) {
    const cudaError_t e =
        cudaFuncSetAttribute(gemm_w8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(W8_SMEM));
    if (e != cudaSuccess) return static_cast<int>(e);
    configured = true;
  }
  quantize_w8_rows_kernel<<<t_pad, 256, 0, stream>>>(x, planes, steps, T, K, t_pad);
  count_launch();
  if (const cudaError_t e = cudaGetLastError()) return static_cast<int>(e);
  const dim3 grid(t_pad / W8_BN, (N + BM - 1) / BM);
  gemm_w8_kernel<<<grid, W8_THREADS, W8_SMEM, stream>>>(map_w, map_p, scales, steps, out, T, N, K, t_pad);
  count_launch();
  return static_cast<int>(cudaGetLastError());
}

}  // namespace tc
}  // namespace kllm

extern "C" int kllm_gemm_w8(const float* x, const int8_t* w, const float* scales, float* out, void* workspace,
                            int n_tokens, int in_dim, int out_dim, void* stream) {
  if (!x || !w || !scales || !out || !workspace || n_tokens <= 0 || in_dim <= 0 || out_dim <= 0) return KLLM_E_INVALID;
  if (in_dim % 64) return KLLM_E_UNSUPPORTED;  // whole 64-groups: one scale per row and group
  // TMA needs 16-byte aligned bases (x is read as float4); scales and out are read / written per element
  if ((reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(w) & 15) ||
      (reinterpret_cast<uintptr_t>(workspace) & 15) || (reinterpret_cast<uintptr_t>(scales) & 3) ||
      (reinterpret_cast<uintptr_t>(out) & 3))
    return KLLM_E_UNSUPPORTED;
  return kllm::tc::launch_w8(x, w, scales, out, workspace, n_tokens, in_dim, out_dim,
                             static_cast<cudaStream_t>(stream));
}

extern "C" int kllm_gemm_tf32(const float* x, const float* w, float* out, int n_tokens, int in_dim, int out_dim,
                              void* stream) {
  if (!x || !w || !out || n_tokens <= 0 || in_dim <= 0 || out_dim <= 0) return KLLM_E_INVALID;
  // TMA needs 16-byte aligned bases and row pitches
  if ((in_dim & 3) || (reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(w) & 15)) return KLLM_E_UNSUPPORTED;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  using namespace kllm::tc;
  if (n_tokens <= 32) return launch<32>(x, w, out, n_tokens, in_dim, out_dim, s);
  if (n_tokens <= 64) return launch<64>(x, w, out, n_tokens, in_dim, out_dim, s);
  if (n_tokens <= 128) return launch<128>(x, w, out, n_tokens, in_dim, out_dim, s);
  return launch<256>(x, w, out, n_tokens, in_dim, out_dim, s);
}
