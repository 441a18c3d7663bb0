// Host-side plumbing shared by the translation units of libkllm_b200.so.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdint>

#include "../../include/kllm_b200.h"

namespace kllm {
// Launch accounting for bench.py's `gpu_launches` claim: every kernel<<<>>> issued by this
// library bumps the counter (graph replays add the node count of the replayed graph).
std::atomic<uint64_t>& launch_counter();
inline void count_launch(uint64_t n = 1) { launch_counter().fetch_add(n, std::memory_order_relaxed); }

// A position that is either a host value or read from device memory at kernel run time; the
// decoder's CUDA graph uses the device form so ONE captured graph serves every position.
struct PosArg {
  const int* ptr;
  int val;
  __host__ __device__ int get() const { return ptr != nullptr ? *ptr : val; }
};

// Output rows of segment s land at seg[s].out + pos * pos_stride[s] (KV-cache rows).
struct GemvExtra {
  PosArg pos{nullptr, 0};
  long long pos_stride[3] = {0, 0, 0};
};

int gemv_dispatch(const kllm_gemv_job* job, const GemvExtra& extra, cudaStream_t stream);
int launch_rope(int flavour, int dim, int kv_dim, int head_size, float* q, float* k_base,
                long long k_pos_stride, PosArg pos, const float* sin_cache,
                const float* cos_cache, cudaStream_t stream);
int launch_mha(PosArg pos, int head_num, int layer_index, int seq_len, int kv_dim, int kv_mul,
               int head_size, float* mha_out, const float* query, float* score,
               const float* key_cache, const float* value_cache, cudaStream_t stream);

// tp_comm.cu: exchange areas [2][world][stride] of 64-bit tagged words, one per rank (peer transport)
int comm_tagged_areas(kllm_comm* comm, unsigned long long** areas8, int* world, int* rank, int* stride);

// prefill.cu: one block of T prompt positions through every layer with batched tcgen05 GEMMs
// (kllm_gemm_tf32 for fp32 weights; kllm_gemm_w8 for int8 group-64 weights when sq..s3 are set)
struct PrefillModel {
  int dim, hidden_dim, layer_num, head_num, kv_head_num, vocab_size, seq_len, head_size, flavour;
  int mega_layout;  // 1: the persistent engine's head-major K / V cache layout (megakernel.cu)
  int attn_split;   // ... whose V rows are cut into attn_split slices of head_size / attn_split dims
  float eps;
  const float* tok_emb;
  const float* const* attn_norm;
  const float* const* ffn_norm;
  const void* const* wq; const void* const* wk; const void* const* wv; const void* const* wo;
  const void* const* w1; const void* const* w2; const void* const* w3;
  // int8 only (NULL for fp32): per-layer scales [rows, in / 64] and the GEMM's activation workspace
  const float* const* sq; const float* const* sk; const float* const* sv; const float* const* so;
  const float* const* s1; const float* const* s2; const float* const* s3;
  void* w8_workspace;
  const float* const* bq; const float* const* bk; const float* const* bv;
  float* key_cache; float* value_cache;
  const float* sin_cache; const float* cos_cache;
};
struct PrefillWorkspace {  // [block, .] activations
  float *x, *xn, *q, *k, *v, *att, *h1, *h3, *tmp;
};
int prefill_block(const PrefillModel& m, PrefillWorkspace& ws, const int32_t* tokens_dev, int T, int start_pos,
                  cudaStream_t stream);
int prefill_attention_smem_opt_in(size_t bytes);

inline float flavour_eps(int flavour) { return flavour == KLLM_FLAVOUR_QWEN2 ? 1e-6f : 1e-5f; }
}  // namespace kllm
