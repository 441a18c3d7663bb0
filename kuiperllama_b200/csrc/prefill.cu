// Batched prompt prefill around the tcgen05 GEMM (prefill_gemm.cu) -- the TOLERANCED alternative to
// feeding the prompt position by position (demo/main.cpp:18-23 calls LLama2Model::predict once per
// prompt token; llama3.cpp:147-167 then runs the whole single-token forward, classifier included).
//
// For a block of T prompt positions every projection is ONE GEMM [T, in] x [out, in]^T on the tensor
// cores (TF32 multiply, fp32 accumulate) instead of T GEMVs, so the weights are streamed once per
// 256 tokens; the small per-token operators (RMSNorm, RoPE, causal attention over the cache, SiLU*gate,
// residual adds) are plain fp32 CUDA kernels over the T rows; only the last position runs the
// classifier (the reference throws the others away, llama3.cpp:738-739).  The K / V rows land in the
// decoder's cache in the layout of the engine that will continue decoding.
//
// Because of TF32 (10 mantissa bits per operand) the cache rows and the final logits agree with the
// position-by-position path to ~1e-3 relative, not bit for bit; tests/test_prefill_gpu.py states the
// bound.  fp32 checkpoints, single GPU.  Int8 (group 64) checkpoints take kllm_gemm_w8 instead (int8 weights
// x 24-bit fixed-point activations, exact integer products): within 1e-4 of the position-by-position path,
// tests/test_prefill_w8_gpu.py.
#include <cuda_runtime.h>

#include <cfloat>
#include <cstdint>

#include "../../include/kllm_b200.h"
#include "kllm_device.cuh"
#include "kllm_host.h"

namespace kllm {
namespace prefill {

__global__ void embed_rows_kernel(const int32_t* __restrict__ tokens, const float* __restrict__ table,
                                  float* __restrict__ x, int dim, int vocab) {
  const int t = blockIdx.x;
  int tok = tokens[t];
  if (tok < 0 || tok >= vocab) tok = 0;
  const float4* src = reinterpret_cast<const float4*>(table + static_cast<size_t>(tok) * dim);
  float4* dst = reinterpret_cast<float4*>(x + static_cast<size_t>(t) * dim);
  for (int i = threadIdx.x; i < (dim >> 2); i += blockDim.x) dst[i] = src[i];
}

__device__ __forceinline__ float block_sum(float v, float* scratch) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(kFull, v, off);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  float total = 0.f;
  for (int w = 0; w < (blockDim.x >> 5); ++w) total += scratch[w];
  return total;
}
__device__ __forceinline__ float block_max(float v, float* scratch) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v = fmaxf(v, __shfl_xor_sync(kFull, v, off));
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  float m = -FLT_MAX;
  for (int w = 0; w < (blockDim.x >> 5); ++w) m = fmaxf(m, scratch[w]);
  return m;
}

// rmsnorm_kernel.cu:4-50 per row (summation order differs: toleranced path)
__global__ void rmsnorm_rows_kernel(const float* __restrict__ x, const float* __restrict__ w, float* __restrict__ out,
                                    int dim, float eps) {
  __shared__ float scratch[32];
  const float* row = x + static_cast<size_t>(blockIdx.x) * dim;
  float* o = out + static_cast<size_t>(blockIdx.x) * dim;
  float ss = 0.f;
  for (int i = threadIdx.x; i < dim; i += blockDim.x) ss += row[i] * row[i];
  const float total = block_sum(ss, scratch);
  const float sc = rsqrtf(total / static_cast<float>(dim) + eps);
  for (int i = threadIdx.x; i < dim; i += blockDim.x) o[i] = (sc * row[i]) * w[i];
}

__global__ void add_bias_rows_kernel(float* __restrict__ y, const float* __restrict__ b, int n) {
  float* row = y + static_cast<size_t>(blockIdx.x) * n;
  for (int i = threadIdx.x; i < n; i += blockDim.x) row[i] += b[i];
}
__global__ void add_rows_kernel(float* __restrict__ x, const float* __restrict__ y, size_t n) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x)
    x[i] = x[i] + y[i];  // llama3.cpp:683,719: x + out
}
__global__ void swiglu_rows_kernel(float* __restrict__ h1, const float* __restrict__ h3, size_t n) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x)
    h1[i] = swiglu_ref(h1[i], h3[i]);
}

struct CacheLayout {
  int mega;  // 1: persistent engine K [kvh][hs/4][seq][4], V [kvh][split][seq][hs/split]; 0: [seq][kv_dim]
  int seq_len, kv_dim, head_size, split;
};
__device__ __forceinline__ size_t k_index(const CacheLayout& c, int pos, int kvh, int i) {
  if (c.mega) return (static_cast<size_t>(kvh) * (c.head_size >> 2) + (i >> 2)) * c.seq_len * 4 + static_cast<size_t>(pos) * 4 + (i & 3);
  return static_cast<size_t>(pos) * c.kv_dim + kvh * c.head_size + i;
}
__device__ __forceinline__ size_t v_index(const CacheLayout& c, int pos, int kvh, int i) {
  if (c.mega) {
    const int dv = c.head_size / c.split;
    return ((static_cast<size_t>(kvh) * c.split + i / dv) * c.seq_len + pos) * dv + i % dv;
  }
  return static_cast<size_t>(pos) * c.kv_dim + kvh * c.head_size + i;
}

// RoPE (rope_kernel.cu) on the T query rows in place, and on the T key rows while they are scattered,
// with the value rows, into the layer's cache.  grid = T, one thread per rotation pair.
__global__ void rope_scatter_kernel(float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                                    const float* __restrict__ sin_t, const float* __restrict__ cos_t,
                                    float* __restrict__ kcache, float* __restrict__ vcache, CacheLayout c, int heads,
                                    int kv_heads, int flavour, int start_pos) {
  const int t = blockIdx.x, pos = start_pos + t, hs = c.head_size, half = hs >> 1;
  float* qrow = q + static_cast<size_t>(t) * heads * hs;
  const float* krow = k + static_cast<size_t>(t) * kv_heads * hs;
  const float* vrow = v + static_cast<size_t>(t) * kv_heads * hs;
  for (int p = threadIdx.x; p < (heads + kv_heads) * half; p += blockDim.x) {
    const int h = p / half, j = p % half;
    int i0, i1;
    if (flavour == KLLM_FLAVOUR_LLAMA2) {
      i0 = 2 * j, i1 = 2 * j + 1;
    } else {
      i0 = j, i1 = j + half;
    }
    const float fci = sin_t[static_cast<size_t>(pos) * hs + 2 * j];
    const float fcr = cos_t[static_cast<size_t>(pos) * hs + 2 * j];
    if (h < heads) {
      float* qh = qrow + h * hs;
      const float a = qh[i0], b = qh[i1];
      qh[i0] = __fmaf_rn(fcr, a, -__fmul_rn(fci, b));
      qh[i1] = __fmaf_rn(fci, a, __fmul_rn(fcr, b));
    } else {
      const int kvh = h - heads;
      const float a = krow[kvh * hs + i0], b = krow[kvh * hs + i1];
      kcache[k_index(c, pos, kvh, i0)] = __fmaf_rn(fcr, a, -__fmul_rn(fci, b));
      kcache[k_index(c, pos, kvh, i1)] = __fmaf_rn(fci, a, __fmul_rn(fcr, b));
    }
  }
  for (int p = threadIdx.x; p < kv_heads * hs; p += blockDim.x)
    vcache[v_index(c, pos, p / hs, p % hs)] = vrow[p];
}

// Causal attention of query (t, head) over cache positions 0 .. start_pos + t (mha_kernel.cu:47-110
// arithmetic, fp32).  grid = (heads, T); scores in dynamic shared memory.
__global__ void attn_rows_kernel(const float* __restrict__ q, const float* __restrict__ kcache,
                                 const float* __restrict__ vcache, float* __restrict__ out, CacheLayout c, int heads,
                                 int kv_mul, int start_pos) {
  extern __shared__ float sc[];
  __shared__ float scratch[32];
  const int head = blockIdx.x, t = blockIdx.y, pos = start_pos + t, hs = c.head_size, kvh = head / kv_mul;
  const float* qh = q + (static_cast<size_t>(t) * heads + head) * hs;
  const float scale = 1.f / sqrtf(static_cast<float>(hs));
  float mx = -FLT_MAX;
  for (int j = threadIdx.x; j <= pos; j += blockDim.x) {
    float s = 0.f;
    for (int i = 0; i < hs; ++i) s = __fmaf_rn(kcache[k_index(c, j, kvh, i)], qh[i], s);
    s *= scale;
    sc[j] = s;
    mx = fmaxf(mx, s);
  }
  mx = block_max(mx, scratch);
  float sum = 0.f;
  for (int j = threadIdx.x; j <= pos; j += blockDim.x) {
    const float e = expf(sc[j] - mx);
    sc[j] = e;
    sum += e;
  }
  sum = block_sum(sum, scratch);
  __syncthreads();
  for (int i = threadIdx.x; i < hs; i += blockDim.x) {
    float acc = 0.f;
    for (int j = 0; j <= pos; ++j) acc = __fmaf_rn(sc[j] / sum, vcache[v_index(c, j, kvh, i)], acc);
    out[(static_cast<size_t>(t) * heads + head) * hs + i] = acc;
  }
}

}  // namespace prefill

using namespace prefill;

#define PF_TRY(expr)                       \
  do {                                     \
    const int rc_ = static_cast<int>(expr); \
    if (rc_ != 0) return rc_;              \
  } while (0)

int prefill_block(const PrefillModel& m, PrefillWorkspace& ws, const int32_t* tokens_dev, int T, int start_pos,
                  cudaStream_t s) {
  const int dim = m.dim, hid = m.hidden_dim, hs = m.head_size, heads = m.head_num, kvh = m.kv_head_num;
  const int q_rows = heads * hs, kvd = kvh * hs;
  const bool w8 = m.sq != nullptr;
  auto gemm = [&](const float* x, const void* w, const float* const* scales, int l, float* out, int K, int N) {
    if (w8) return kllm_gemm_w8(x, static_cast<const int8_t*>(w), scales[l], out, m.w8_workspace, T, K, N, s);
    return kllm_gemm_tf32(x, static_cast<const float*>(w), out, T, K, N, s);
  };
  auto count = [&]() {
    count_launch();
    return static_cast<int>(cudaGetLastError());
  };
  const int ew_grid = 592;  // 4 x 148 SMs for the grid-stride elementwise kernels
  embed_rows_kernel<<<T, 256, 0, s>>>(tokens_dev, m.tok_emb, ws.x, dim, m.vocab_size);
  PF_TRY(count());
  const CacheLayout cl{m.mega_layout, m.seq_len, kvd, hs, m.attn_split > 0 ? m.attn_split : 1};
  for (int l = 0; l < m.layer_num; ++l) {
    const size_t layer_off = static_cast<size_t>(l) * m.seq_len * kvd;
    rmsnorm_rows_kernel<<<T, 256, 0, s>>>(ws.x, m.attn_norm[l], ws.xn, dim, m.eps);
    PF_TRY(count());
    PF_TRY(gemm(ws.xn, m.wq[l], m.sq, l, ws.q, dim, q_rows));
    PF_TRY(gemm(ws.xn, m.wk[l], m.sk, l, ws.k, dim, kvd));
    PF_TRY(gemm(ws.xn, m.wv[l], m.sv, l, ws.v, dim, kvd));
    if (m.bq != nullptr) {
      add_bias_rows_kernel<<<T, 256, 0, s>>>(ws.q, m.bq[l], q_rows);
      add_bias_rows_kernel<<<T, 256, 0, s>>>(ws.k, m.bk[l], kvd);
      add_bias_rows_kernel<<<T, 256, 0, s>>>(ws.v, m.bv[l], kvd);
      count_launch(2);
      PF_TRY(count());
    }
    rope_scatter_kernel<<<T, 256, 0, s>>>(ws.q, ws.k, ws.v, m.sin_cache, m.cos_cache, m.key_cache + layer_off,
                                          m.value_cache + layer_off, cl, heads, kvh, m.flavour, start_pos);
    PF_TRY(count());
    const size_t sc_bytes = static_cast<size_t>(start_pos + T) * sizeof(float);
    attn_rows_kernel<<<dim3(heads, T), 128, sc_bytes, s>>>(ws.q, m.key_cache + layer_off, m.value_cache + layer_off,
                                                           ws.att, cl, heads, heads / kvh, start_pos);
    PF_TRY(count());
    PF_TRY(gemm(ws.att, m.wo[l], m.so, l, ws.tmp, q_rows, dim));
    add_rows_kernel<<<ew_grid, 256, 0, s>>>(ws.x, ws.tmp, static_cast<size_t>(T) * dim);
    PF_TRY(count());
    rmsnorm_rows_kernel<<<T, 256, 0, s>>>(ws.x, m.ffn_norm[l], ws.xn, dim, m.eps);
    PF_TRY(count());
    PF_TRY(gemm(ws.xn, m.w1[l], m.s1, l, ws.h1, dim, hid));
    PF_TRY(gemm(ws.xn, m.w3[l], m.s3, l, ws.h3, dim, hid));
    swiglu_rows_kernel<<<ew_grid, 256, 0, s>>>(ws.h1, ws.h3, static_cast<size_t>(T) * hid);
    PF_TRY(count());
    PF_TRY(gemm(ws.h1, m.w2[l], m.s2, l, ws.tmp, hid, dim));
    add_rows_kernel<<<ew_grid, 256, 0, s>>>(ws.x, ws.tmp, static_cast<size_t>(T) * dim);
    PF_TRY(count());
  }
  return 0;
}

int prefill_attention_smem_opt_in(size_t bytes) {
  static size_t configured = 0;
  if (bytes <= 48 * 1024 || bytes <= configured) return 0;
  const cudaError_t e =
      cudaFuncSetAttribute(attn_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes));
  if (e != cudaSuccess) return static_cast<int>(e);
  configured = bytes;
  return 0;
}

}  // namespace kllm
