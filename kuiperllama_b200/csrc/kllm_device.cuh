// Device-side helpers shared by the sm_100a kernels.
//
// "Reference order" below always means the floating-point operation order of the reference's
// own CUDA kernels as compiled by nvcc 12.9 for sm_100a (read off the SASS of oracle/_ref,
// see DESIGN.md "Bit-exactness").  All arithmetic that must match is written with explicit
// round-to-nearest intrinsics so the compiler can neither fuse nor split it differently.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace kllm {

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

// 128-bit streaming load: read-only path, do not allocate in L1 (weights are touched once).
__device__ __forceinline__ float4 ldg_stream_f4(const float4* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p));
  return v;
}

__device__ __forceinline__ uint32_t ldg_stream_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}

// matmul_kernel.cu:30-34 as compiled: part = fma(x.w,w.w, fma(x.z,w.z, fma(x.x,w.x, x.y*w.y))).
__device__ __forceinline__ float dot4_ref(const float4& x, const float4& w) {
  float p = __fmul_rn(x.y, w.y);
  p = __fmaf_rn(x.x, w.x, p);
  p = __fmaf_rn(x.z, w.z, p);
  p = __fmaf_rn(x.w, w.w, p);
  return p;
}

// cub::WarpReduce shuffle-down tree (offsets 1,2,4,8,16).  cub only adds when the source lane
// is in range; adding unconditionally changes upper lanes only, never lane 0's result.
__device__ __forceinline__ float warp_tree_sum(float v) {
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) v = __fadd_rn(v, __shfl_down_sync(kFull, v, off));
  return v;
}

// cub::BlockReduce<float,128>::Sum (BLOCK_REDUCE_WARP_REDUCTIONS) over 128 virtual threads laid
// out as acc[j] = virtual thread (lane + 32*j): per-virtual-warp shuffle tree, then
// ((w0+w1)+w2)+w3.  Result valid in lane 0.
__device__ __forceinline__ float block128_sum_vt(const float acc[4]) {
  const float a0 = warp_tree_sum(acc[0]);
  const float a1 = warp_tree_sum(acc[1]);
  const float a2 = warp_tree_sum(acc[2]);
  const float a3 = warp_tree_sum(acc[3]);
  return __fadd_rn(__fadd_rn(__fadd_rn(a0, a1), a2), a3);
}

// Same reduction for the layout acc[e] = virtual thread (4*lane + e): a virtual warp is 8
// consecutive lanes x 4 registers.  Result valid in lane 0.
__device__ __forceinline__ float block128_sum_quad(const float acc[4]) {
  float v0 = acc[0], v1 = acc[1], v2 = acc[2], v3 = acc[3];
  // offset 1
  float n0 = __shfl_down_sync(kFull, v0, 1);
  float t0 = __fadd_rn(v0, v1), t1 = __fadd_rn(v1, v2), t2 = __fadd_rn(v2, v3),
        t3 = __fadd_rn(v3, n0);
  v0 = t0, v1 = t1, v2 = t2, v3 = t3;
  // offset 2
  n0 = __shfl_down_sync(kFull, v0, 1);
  float n1 = __shfl_down_sync(kFull, v1, 1);
  t0 = __fadd_rn(v0, v2), t1 = __fadd_rn(v1, v3), t2 = __fadd_rn(v2, n0), t3 = __fadd_rn(v3, n1);
  v0 = t0, v1 = t1, v2 = t2, v3 = t3;
  // offsets 4, 8, 16 (= 1, 2, 4 lanes); only element 0 feeds virtual lane 0 from here on
  v0 = __fadd_rn(v0, __shfl_down_sync(kFull, v0, 1));
  v0 = __fadd_rn(v0, __shfl_down_sync(kFull, v0, 2));
  v0 = __fadd_rn(v0, __shfl_down_sync(kFull, v0, 4));
  const float a1 = __shfl_sync(kFull, v0, 8);
  const float a2 = __shfl_sync(kFull, v0, 16);
  const float a3 = __shfl_sync(kFull, v0, 24);
  return __fadd_rn(__fadd_rn(__fadd_rn(v0, a1), a2), a3);
}

// The two reductions above, "packed": only lane 0's value of the cub tree is ever used, and that
// value is the balanced binary tree over the 32 lanes (adjacent pairs first), so lanes may trade
// accumulators instead of all reducing all four: after the offset-1 step every lane carries two of
// the four virtual warps, after offset 2 one.  Every addition has the same two operands as in
// cub's tree (FADD commutes), so the result is bit-identical; 10 shuffles + 9 adds instead of
// 20 + 23.  The total is returned in EVERY lane.
__device__ __forceinline__ float block128_sum_vt_packed(const float acc[4], int lane) {
  const bool odd = lane & 1;
  // offset 1: even lanes keep virtual warps 0,1 -- odd lanes 2,3
  const float k0 = odd ? acc[2] : acc[0], k1 = odd ? acc[3] : acc[1];
  const float g0 = odd ? acc[0] : acc[2], g1 = odd ? acc[1] : acc[3];
  const float s0 = __fadd_rn(k0, __shfl_xor_sync(kFull, g0, 1));
  const float s1 = __fadd_rn(k1, __shfl_xor_sync(kFull, g1, 1));
  // offset 2: bit 1 of the lane picks which of the two survives
  const bool hi = lane & 2;
  float v = __fadd_rn(hi ? s1 : s0, __shfl_xor_sync(kFull, hi ? s0 : s1, 2));
  v = __fadd_rn(v, __shfl_xor_sync(kFull, v, 4));
  v = __fadd_rn(v, __shfl_xor_sync(kFull, v, 8));
  v = __fadd_rn(v, __shfl_xor_sync(kFull, v, 16));
  // lanes == 0,2,1,3 (mod 4) now hold virtual warps 0,1,2,3
  const float a0 = __shfl_sync(kFull, v, 0), a1 = __shfl_sync(kFull, v, 2);
  const float a2 = __shfl_sync(kFull, v, 1), a3 = __shfl_sync(kFull, v, 3);
  return __fadd_rn(__fadd_rn(__fadd_rn(a0, a1), a2), a3);
}

// acc[e] = virtual thread (4*lane + e): offsets 1 and 2 of the tree are lane-local, offsets 4, 8,
// 16 are lane distances 1, 2, 4 inside each group of 8 lanes (= one virtual warp).
__device__ __forceinline__ float block128_sum_quad_packed(const float acc[4]) {
  float v = __fadd_rn(__fadd_rn(acc[0], acc[1]), __fadd_rn(acc[2], acc[3]));
  v = __fadd_rn(v, __shfl_xor_sync(kFull, v, 1));
  v = __fadd_rn(v, __shfl_xor_sync(kFull, v, 2));
  v = __fadd_rn(v, __shfl_xor_sync(kFull, v, 4));
  const float a0 = __shfl_sync(kFull, v, 0), a1 = __shfl_sync(kFull, v, 8);
  const float a2 = __shfl_sync(kFull, v, 16), a3 = __shfl_sync(kFull, v, 24);
  return __fadd_rn(__fadd_rn(__fadd_rn(a0, a1), a2), a3);
}

// Exact int8 -> fp32 for the four bytes of `packed` without the slow I2F pipe:
// (b ^ 0x80) dropped into the mantissa of 2^23 gives 2^23 + b + 128; subtracting
// 2^23 + 128 is exact.  Equal to static_cast<float>(int8) (matmul_kernel.cu:73).
__device__ __forceinline__ void int8x4_to_float(uint32_t packed, float out[4]) {
  const uint32_t t = packed ^ 0x80808080u;
  const float magic = 8388736.0f;  // 2^23 + 128
  out[0] = __fsub_rn(__uint_as_float(__byte_perm(t, 0x4B000000u, 0x7650)), magic);
  out[1] = __fsub_rn(__uint_as_float(__byte_perm(t, 0x4B000000u, 0x7651)), magic);
  out[2] = __fsub_rn(__uint_as_float(__byte_perm(t, 0x4B000000u, 0x7652)), magic);
  out[3] = __fsub_rn(__uint_as_float(__byte_perm(t, 0x4B000000u, 0x7653)), magic);
}

// Fixed-point form of one 64-element activation group for the int8 x int8 paths (the fast decode
// mode's dp4a / mma.sync rows, megakernel.cu, and the kind::i8 prompt GEMM, prefill_gemm.cu):
//     x_i ~= step * q_i,  step = gmax * 2^-22,  q_i = rint(x_i * (2^22 / gmax)),  |q_i| <= 2^22,
// q_i split into three balanced base-256 digits, q = 65536 a2 + 256 a1 + a0, each in int8.  An all-zero
// group has step 0 and digits 0.  This is the ONE definition both kernels use.
__device__ __forceinline__ float w8_group_step(float gmax) { return gmax * (1.0f / 4194304.0f); }  // 2^-22
__device__ __forceinline__ float w8_group_inv(float gmax) { return gmax > 0.f ? 4194304.0f / gmax : 0.f; }
// four values -> one packed word (byte b = element b) of each digit plane
__device__ __forceinline__ void w8_digits4(const float (&e)[4], float inv, uint32_t& p0, uint32_t& p1,
                                           uint32_t& p2) {
  p0 = 0, p1 = 0, p2 = 0;
#pragma unroll
  for (int b = 0; b < 4; ++b) {
    const int qv = __float2int_rn(e[b] * inv);  // |qv| <= 2^22
    const int a0 = ((qv + 128) & 255) - 128;    // balanced digits: qv = 65536 a2 + 256 a1 + a0
    const int q1 = (qv - a0) >> 8;
    const int a1 = ((q1 + 128) & 255) - 128;
    const int a2 = (q1 - a1) >> 8;
    p0 |= static_cast<uint32_t>(a0 & 255) << (8 * b);
    p1 |= static_cast<uint32_t>(a1 & 255) << (8 * b);
    p2 |= static_cast<uint32_t>(a2 & 255) << (8 * b);
  }
}

// swiglu_kernel.cu:16-19: value = 1/(1+exp(-a)); (a*value)*b.  Written with plain operators
// on purpose: the reference build contracts expf's final scale multiply with the "1.0f +"
// (SASS: MUFU.EX2; FFMA r, s, e, 1.0), and the same source form makes nvcc do the same here.
__device__ __forceinline__ float swiglu_ref(float a, float b) {
  float value = 1.0f / (1.0f + exp(-a));
  a = a * value;
  return a * b;
}

}  // namespace kllm
