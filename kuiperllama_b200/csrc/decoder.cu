// Device-resident single-batch decoder: the per-token forward of LLama2Model / Qwen2Model
// (kuiper/source/model/llama3.cpp:147-167, 600-745; qwen2.cpp) as a fixed chain of fused
// launches captured ONCE in a CUDA graph and replayed for every position.
//
//   reference, per layer (15-18 launches)          here (6 launches)
//   rmsnorm, wq, wk, wv [+3 bias adds]        ->   gemv_fused(norm -> q | k@cache | v@cache [+bias])
//   rope (pos read on the host)               ->   rope (pos read from device memory)
//   mha                                       ->   mha
//   wo, add                                   ->   gemv_fused(wo, + residual)
//   rmsnorm, w1, w3, swiglu                   ->   gemv_fused(norm -> w1|w3 -> silu*gate)
//   w2, add                                   ->   gemv_fused(w2, + residual)
//   final: rmsnorm, cls, argmax(+malloc+sync) ->   gemv_fused(norm -> cls), argmax+advance
//
// The position, the current token and the step counter live in device memory, so the
// captured graph is position independent and a whole greedy run needs no host round trip
// (reference: 2 blocking copies + 1 cudaMalloc per token, emb_kernel.cu:25-29,
// argmax_kernel.cu:73-87).  Buffer roles follow llama3.cpp:425-500.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../include/kllm_b200.h"
#include "kllm_device.cuh"
#include "kllm_host.h"
#include "megakernel.h"

namespace kllm {

struct StepState {  // device-resident loop state
  int32_t token;    // input token of the current step
  int32_t pos;      // position of the current step
  int32_t step;     // steps done since generate() started
  int32_t next;     // greedy id produced by the last step
};

__global__ void embed_token_kernel(const StepState* st, const float* __restrict__ table,
                                   float* x, int dim, int vocab) {
  const int32_t token = st->token;
  if (token < 0 || token >= vocab) return;
  const float4* s4 = reinterpret_cast<const float4*>(table + static_cast<size_t>(token) * dim);
  float4* d4 = reinterpret_cast<float4*>(x);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < (dim >> 2); i += gridDim.x * blockDim.x)
    d4[i] = s4[i];
}

// Greedy argmax (argmax_kernel.cu:49-71 semantics: max value, lowest index) fused with the
// loop bookkeeping: record the id, feed it (or the teacher's id) to the next step, pos += 1.
__global__ void __launch_bounds__(1024)
argmax_advance_kernel(const float* __restrict__ logits, int n, StepState* st, int32_t* out_tokens,
                      const int32_t* teacher, int max_steps) {
  __shared__ float sv[32];
  __shared__ int si[32];
  float bv = 0.f;
  int bi = -1;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float v = logits[i];
    if (bi < 0 || v > bv) {
      bv = v;
      bi = i;
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  auto fold = [](float& v, int& i, float ov, int oi) {
    if (oi >= 0 && (i < 0 || ov > v || (ov == v && oi < i))) {
      v = ov;
      i = oi;
    }
  };
#pragma unroll
  for (int off = 16; off > 0; off >>= 1)
    fold(bv, bi, __shfl_down_sync(kFull, bv, off), __shfl_down_sync(kFull, bi, off));
  if (lane == 0) {
    sv[warp] = bv;
    si[warp] = bi;
  }
  __syncthreads();
  if (warp == 0) {
    bv = sv[lane];
    bi = si[lane];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1)
      fold(bv, bi, __shfl_down_sync(kFull, bv, off), __shfl_down_sync(kFull, bi, off));
    if (lane == 0) {
      const int next = bi < 0 ? 0 : bi;
      const int step = st->step;
      st->next = next;
      if (out_tokens != nullptr && step < max_steps) out_tokens[step] = next;
      st->token = (teacher != nullptr && step + 1 < max_steps) ? teacher[step + 1] : next;
      st->pos = st->pos + 1;
      st->step = step + 1;
    }
  }
}

}  // namespace kllm

using namespace kllm;

struct kllm_decoder {
  kllm_decoder_desc d{};
  std::vector<const float*> attn_norm, ffn_norm;
  std::vector<const void*> wq, wk, wv, wo, w1, w2, w3;
  std::vector<const float*> sq, sk, sv, so, s1, s2, s3, bq, bk, bv;
  int kv_dim = 0, kv_mul = 0, head_size = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  // device buffers
  float *x = nullptr, *q = nullptr, *attn = nullptr, *h = nullptr, *logits = nullptr;
  float *score = nullptr, *kcache = nullptr, *vcache = nullptr, *sin_t = nullptr, *cos_t = nullptr;
  float* tp_tmp = nullptr;
  float* k_raw = nullptr;  // persistent engine: un-rotated key row of the current position
  MegaEngine mega;
  bool use_mega = false;
  StepState* st = nullptr;
  int32_t* out_tokens = nullptr;  // device [seq_len]
  int32_t* teacher = nullptr;     // device [seq_len]
  StepState* st_host = nullptr;   // pinned
  int32_t* io_host = nullptr;     // pinned scratch
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;       // out_tokens recorded, no teacher
  cudaGraph_t graph_tf = nullptr;
  cudaGraphExec_t exec_tf = nullptr;    // teacher forced
  int launches_per_step = 0;
  // batched tcgen05 prefill (kllm_decoder_prefill_tf32): activations of one block of prompt positions
  float* pf_buf = nullptr;
  PrefillWorkspace pf_ws{};
  void* pf_w8_ws = nullptr;  // kllm_decoder_prefill_w8: kllm_gemm_w8's activation workspace
};

namespace {

#define KLLM_TRY(expr)                      \
  do {                                      \
    const int rc_ = static_cast<int>(expr); \
    if (rc_ != 0) return rc_;               \
  } while (0)

template <typename T>
std::vector<T> copy_ptrs(const T* src, int n) {
  std::vector<T> v;
  if (src != nullptr) v.assign(src, src + n);
  return v;
}

// x += all-reduce(tp_tmp): the row-parallel matmul's partial sums meet here (SURVEY.md 8e)
int tp_reduce_into_x(kllm_decoder* dc, cudaStream_t s) {
  const kllm_decoder_desc& d = dc->d;
  if (d.comm != nullptr) return kllm_comm_allreduce_residual(d.comm, dc->tp_tmp, dc->x, dc->x, d.dim, s);
  KLLM_TRY(d.allreduce(d.allreduce_ctx, dc->tp_tmp, d.dim, s));
  return kllm_add_f32(dc->x, dc->tp_tmp, dc->x, d.dim, s);
}

int enqueue_step(kllm_decoder* dc, bool with_teacher, cudaStream_t s) {
  const kllm_decoder_desc& d = dc->d;
  const int dim = d.dim, L = d.layer_num, hid = d.hidden_dim;
  const int q_rows = d.head_num * dc->head_size;  // == dim unless tensor-parallel
  const int kvd = dc->kv_dim;
  const float eps = flavour_eps(d.flavour);
  const PosArg pos{&dc->st->pos, 0};
  const bool tp = d.tp_size > 1;
  const uint64_t before = launch_counter().load();

  embed_token_kernel<<<4, 256, 0, s>>>(dc->st, d.tok_emb, dc->x, dim, d.vocab_size);
  count_launch();
  KLLM_TRY(cudaGetLastError());

  for (int l = 0; l < L; ++l) {
    const size_t layer_off = static_cast<size_t>(l) * d.seq_len * kvd;
    // attention_rms + attention_qkv (llama3.cpp:600-640); k, v go straight into the cache row
    {
      kllm_gemv_job j{};
      j.x = dc->x;
      j.norm_w = dc->attn_norm[l];
      j.norm_eps = eps;
      j.in_dim = dim;
      j.group_size = d.group_size;
      j.n_seg = 3;
      j.seg[0] = {dc->wq[l], d.group_size ? dc->sq[l] : nullptr, dc->bq.empty() ? nullptr : dc->bq[l],
                  dc->q, q_rows};
      j.seg[1] = {dc->wk[l], d.group_size ? dc->sk[l] : nullptr, dc->bk.empty() ? nullptr : dc->bk[l],
                  dc->kcache + layer_off, kvd};
      j.seg[2] = {dc->wv[l], d.group_size ? dc->sv[l] : nullptr, dc->bv.empty() ? nullptr : dc->bv[l],
                  dc->vcache + layer_off, kvd};
      GemvExtra ex;
      ex.pos = pos;
      ex.pos_stride[1] = kvd;
      ex.pos_stride[2] = kvd;
      KLLM_TRY(gemv_dispatch(&j, ex, s));
    }
    KLLM_TRY(launch_rope(d.flavour, q_rows, kvd, dc->head_size, dc->q, dc->kcache + layer_off, kvd,
                         pos, dc->sin_t, dc->cos_t, s));
    // attention_mha (llama3.cpp:652-676)
    KLLM_TRY(launch_mha(pos, d.head_num, l, d.seq_len, kvd, dc->kv_mul, dc->head_size, dc->attn,
                        dc->q, dc->score, dc->kcache, dc->vcache, s));
    {
      kllm_gemv_job j{};
      j.x = dc->attn;
      j.in_dim = q_rows;
      j.group_size = d.group_size;
      j.n_seg = 1;
      j.seg[0] = {dc->wo[l], d.group_size ? dc->so[l] : nullptr, nullptr, tp ? dc->tp_tmp : dc->x, dim};
      j.residual = tp ? nullptr : dc->x;  // feed_forward's first add (llama3.cpp:683-684)
      KLLM_TRY(gemv_dispatch(&j, GemvExtra{}, s));
      if (tp) KLLM_TRY(tp_reduce_into_x(dc, s));
    }
    // feed_forward (llama3.cpp:686-720)
    {
      kllm_gemv_job j{};
      j.x = dc->x;
      j.norm_w = dc->ffn_norm[l];
      j.norm_eps = eps;
      j.in_dim = dim;
      j.group_size = d.group_size;
      j.n_seg = 2;
      j.seg[0] = {dc->w1[l], d.group_size ? dc->s1[l] : nullptr, nullptr, dc->h, hid};
      j.seg[1] = {dc->w3[l], d.group_size ? dc->s3[l] : nullptr, nullptr, nullptr, hid};
      j.swiglu_pair = 1;
      KLLM_TRY(gemv_dispatch(&j, GemvExtra{}, s));
    }
    {
      kllm_gemv_job j{};
      j.x = dc->h;
      j.in_dim = hid;
      j.group_size = d.group_size;
      j.n_seg = 1;
      j.seg[0] = {dc->w2[l], d.group_size ? dc->s2[l] : nullptr, nullptr, tp ? dc->tp_tmp : dc->x, dim};
      j.residual = tp ? nullptr : dc->x;
      KLLM_TRY(gemv_dispatch(&j, GemvExtra{}, s));
      if (tp) KLLM_TRY(tp_reduce_into_x(dc, s));
    }
  }
  // cls_logits (llama3.cpp:722-731) + post_processing (:733-745)
  {
    kllm_gemv_job j{};
    j.x = dc->x;
    j.norm_w = d.final_norm;
    j.norm_eps = eps;
    j.in_dim = dim;
    j.group_size = d.group_size;
    j.n_seg = 1;
    j.seg[0] = {d.wcls, d.group_size ? d.scls : nullptr, nullptr, dc->logits, d.vocab_size};
    KLLM_TRY(gemv_dispatch(&j, GemvExtra{}, s));
  }
  argmax_advance_kernel<<<1, 1024, 0, s>>>(dc->logits, d.vocab_size, dc->st, dc->out_tokens,
                                           with_teacher ? dc->teacher : nullptr, d.seq_len);
  count_launch();
  KLLM_TRY(cudaGetLastError());
  dc->launches_per_step = static_cast<int>(launch_counter().load() - before);
  return 0;
}

int capture(kllm_decoder* dc, bool with_teacher, cudaGraph_t* graph, cudaGraphExec_t* exec) {
  KLLM_TRY(cudaStreamBeginCapture(dc->stream, cudaStreamCaptureModeRelaxed));
  const int rc = enqueue_step(dc, with_teacher, dc->stream);
  cudaGraph_t g = nullptr;
  const cudaError_t end = cudaStreamEndCapture(dc->stream, &g);
  if (rc != 0) {
    if (g) cudaGraphDestroy(g);
    return rc;
  }
  KLLM_TRY(end);
  *graph = g;
  KLLM_TRY(cudaGraphInstantiate(exec, g, 0));
  // capturing does not execute: undo the launch accounting of the capture pass
  launch_counter().fetch_sub(static_cast<uint64_t>(dc->launches_per_step));
  return 0;
}

}  // namespace

extern "C" {

int kllm_decoder_create(const kllm_decoder_desc* desc, void* stream, kllm_decoder** out) {
  if (!desc || !out) return KLLM_E_INVALID;
  const kllm_decoder_desc& d = *desc;
  if (d.dim <= 0 || d.hidden_dim <= 0 || d.layer_num <= 0 || d.head_num <= 0 ||
      d.kv_head_num <= 0 || d.vocab_size <= 0 || d.seq_len <= 0)
    return KLLM_E_INVALID;
  if (!d.tok_emb || !d.attn_norm || !d.ffn_norm || !d.final_norm || !d.wq || !d.wk || !d.wv ||
      !d.wo || !d.w1 || !d.w2 || !d.w3 || !d.wcls)
    return KLLM_E_INVALID;
  if (d.group_size > 0 && (!d.sq || !d.sk || !d.sv || !d.so || !d.s1 || !d.s2 || !d.s3 || !d.scls))
    return KLLM_E_INVALID;
  const int tp = d.tp_size > 1 ? d.tp_size : 1;
  if (tp > 1 && d.allreduce == nullptr && d.comm == nullptr) return KLLM_E_INVALID;
  // head_size from the FULL model: dim / (head_num * tp)
  if (d.dim % (d.head_num * tp) != 0 || d.head_num % d.kv_head_num != 0) return KLLM_E_INVALID;
  if ((d.dim & 3) != 0 || (d.hidden_dim & 3) != 0) return KLLM_E_UNSUPPORTED;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return KLLM_E_NODEVICE;

  auto* dc = new kllm_decoder();
  dc->d = d;
  const int L = d.layer_num;
  dc->attn_norm = copy_ptrs(d.attn_norm, L);
  dc->ffn_norm = copy_ptrs(d.ffn_norm, L);
  dc->wq = copy_ptrs(d.wq, L), dc->wk = copy_ptrs(d.wk, L), dc->wv = copy_ptrs(d.wv, L);
  dc->wo = copy_ptrs(d.wo, L), dc->w1 = copy_ptrs(d.w1, L), dc->w2 = copy_ptrs(d.w2, L);
  dc->w3 = copy_ptrs(d.w3, L);
  if (d.group_size > 0) {
    dc->sq = copy_ptrs(d.sq, L), dc->sk = copy_ptrs(d.sk, L), dc->sv = copy_ptrs(d.sv, L);
    dc->so = copy_ptrs(d.so, L), dc->s1 = copy_ptrs(d.s1, L), dc->s2 = copy_ptrs(d.s2, L);
    dc->s3 = copy_ptrs(d.s3, L);
  }
  dc->bq = copy_ptrs(d.bq, L), dc->bk = copy_ptrs(d.bk, L), dc->bv = copy_ptrs(d.bv, L);
  dc->head_size = d.dim / (d.head_num * tp);
  dc->kv_dim = d.kv_head_num * dc->head_size;
  dc->kv_mul = d.head_num / d.kv_head_num;
  dc->d.tp_size = tp;

  if (stream != nullptr) {
    dc->stream = static_cast<cudaStream_t>(stream);
  } else {
    if (cudaStreamCreateWithFlags(&dc->stream, cudaStreamNonBlocking) != cudaSuccess) {
      delete dc;
      return KLLM_E_NODEVICE;
    }
    dc->own_stream = true;
    // A private non-blocking stream does not order against the legacy default stream: weights the
    // caller uploaded or produced there (or anywhere else) must have landed before the first launch.
    if (cudaDeviceSynchronize() != cudaSuccess) {
      cudaStreamDestroy(dc->stream);
      delete dc;
      return KLLM_E_NODEVICE;
    }
  }

  auto fail = [&](int rc) {
    kllm_decoder_destroy(dc);
    return rc;
  };
  auto dev_alloc = [&](float** p, size_t n) {
    if (cudaMalloc(p, n * sizeof(float)) != cudaSuccess) return 1;
    return static_cast<int>(cudaMemsetAsync(*p, 0, n * sizeof(float), dc->stream));
  };
  const size_t kv_elems = static_cast<size_t>(L) * d.seq_len * dc->kv_dim;
  const int q_rows = d.head_num * dc->head_size;
  if (dev_alloc(&dc->x, d.dim) || dev_alloc(&dc->q, q_rows) || dev_alloc(&dc->attn, q_rows) ||
      dev_alloc(&dc->h, d.hidden_dim) || dev_alloc(&dc->logits, d.vocab_size) ||
      dev_alloc(&dc->score, static_cast<size_t>(d.head_num) * d.seq_len) ||
      dev_alloc(&dc->kcache, kv_elems) || dev_alloc(&dc->vcache, kv_elems) ||
      dev_alloc(&dc->sin_t, static_cast<size_t>(d.seq_len) * dc->head_size) ||
      dev_alloc(&dc->cos_t, static_cast<size_t>(d.seq_len) * dc->head_size) ||
      dev_alloc(&dc->tp_tmp, d.dim) || dev_alloc(&dc->k_raw, dc->kv_dim))
    return fail(static_cast<int>(cudaErrorMemoryAllocation));
  if (cudaMalloc(&dc->st, sizeof(StepState)) != cudaSuccess ||
      cudaMalloc(&dc->out_tokens, sizeof(int32_t) * d.seq_len) != cudaSuccess ||
      cudaMalloc(&dc->teacher, sizeof(int32_t) * d.seq_len) != cudaSuccess ||
      cudaMallocHost(&dc->st_host, sizeof(StepState)) != cudaSuccess ||
      cudaMallocHost(&dc->io_host, sizeof(int32_t) * d.seq_len) != cudaSuccess)
    return fail(static_cast<int>(cudaErrorMemoryAllocation));
  cudaMemsetAsync(dc->st, 0, sizeof(StepState), dc->stream);

  int rc = kllm_sincos_init(dc->head_size, d.seq_len, d.flavour, dc->sin_t, dc->cos_t, dc->stream);
  if (rc != 0) return fail(rc);
  // Engine: the persistent megakernel (one cooperative launch per run) when the shape fits its
  // shared-memory ring, else the CUDA-graph chain of fused launches.  KLLM_ENGINE=graph|persistent
  // forces one (persistent fails loudly if unsupported).  Both are CUDA; neither is a fallback to
  // anything off-device.
  const char* want = getenv("KLLM_ENGINE");
  const bool force_graph = want != nullptr && strcmp(want, "graph") == 0;
  const bool force_mega = want != nullptr && strcmp(want, "persistent") == 0;
  // tensor parallel: the persistent engine needs the peer-memory transport (its exchange IS
  // the all-reduce); with NCCL or a caller-supplied callback the graph engine is used
  unsigned long long* tp_areas[8] = {};
  int tp_world = 1, tp_rank = 0, tp_stride = 0;
  bool mega_ok = tp == 1;
  if (tp > 1 && d.comm != nullptr &&
      comm_tagged_areas(d.comm, tp_areas, &tp_world, &tp_rank, &tp_stride) == 0 && tp_world == tp &&
      tp_stride >= d.dim)
    mega_ok = true;
  if (!force_graph && mega_ok) {
    MegaModel mm{};
    mm.tp_world = tp, mm.tp_rank = tp_rank, mm.tp_stride = tp_stride;
    mm.numerics = d.numerics;
    for (int r = 0; r < 8; ++r) mm.tp_data[r] = tp_areas[r];
    mm.dim = d.dim, mm.hidden_dim = d.hidden_dim, mm.layer_num = L, mm.head_num = d.head_num;
    mm.kv_head_num = d.kv_head_num, mm.vocab_size = d.vocab_size, mm.seq_len = d.seq_len;
    mm.head_size = dc->head_size, mm.kv_dim = dc->kv_dim, mm.kv_mul = dc->kv_mul;
    mm.flavour = d.flavour, mm.group_size = d.group_size;
    mm.tok_emb = d.tok_emb, mm.attn_norm = dc->attn_norm.data(), mm.ffn_norm = dc->ffn_norm.data();
    mm.final_norm = d.final_norm;
    mm.wq = dc->wq.data(), mm.wk = dc->wk.data(), mm.wv = dc->wv.data(), mm.wo = dc->wo.data();
    mm.w1 = dc->w1.data(), mm.w2 = dc->w2.data(), mm.w3 = dc->w3.data(), mm.wcls = d.wcls;
    if (d.group_size > 0) {
      mm.sq = dc->sq.data(), mm.sk = dc->sk.data(), mm.sv = dc->sv.data(), mm.so = dc->so.data();
      mm.s1 = dc->s1.data(), mm.s2 = dc->s2.data(), mm.s3 = dc->s3.data(), mm.scls = d.scls;
    }
    mm.bq = dc->bq.empty() ? nullptr : dc->bq.data();
    mm.bk = dc->bk.empty() ? nullptr : dc->bk.data();
    mm.bv = dc->bv.empty() ? nullptr : dc->bv.data();
    mm.x = dc->x, mm.q = dc->q, mm.k_raw = dc->k_raw, mm.attn_out = dc->attn, mm.h = dc->h;
    mm.logits = dc->logits, mm.score = dc->score, mm.key_cache = dc->kcache, mm.value_cache = dc->vcache;
    mm.sin_cache = dc->sin_t, mm.cos_cache = dc->cos_t, mm.state = dc->st, mm.out_tokens = dc->out_tokens;
    rc = dc->mega.init(mm, dc->stream);
    if (rc == 0) {
      dc->use_mega = true;
      dc->launches_per_step = 1;
    } else if (rc != KLLM_E_UNSUPPORTED || force_mega) {
      return fail(rc);
    }
  } else if (force_mega) {
    return fail(KLLM_E_UNSUPPORTED);
  }
  if (!dc->use_mega) {
    if ((rc = capture(dc, false, &dc->graph, &dc->exec)) != 0) return fail(rc);
    if ((rc = capture(dc, true, &dc->graph_tf, &dc->exec_tf)) != 0) return fail(rc);
  }
  if (cudaStreamSynchronize(dc->stream) != cudaSuccess) return fail(static_cast<int>(cudaGetLastError()));
  *out = dc;
  return 0;
}

void kllm_decoder_destroy(kllm_decoder* dc) {
  if (!dc) return;
  if (dc->stream) cudaStreamSynchronize(dc->stream);
  dc->mega.destroy();
  if (dc->exec) cudaGraphExecDestroy(dc->exec);
  if (dc->graph) cudaGraphDestroy(dc->graph);
  if (dc->exec_tf) cudaGraphExecDestroy(dc->exec_tf);
  if (dc->graph_tf) cudaGraphDestroy(dc->graph_tf);
  float* bufs[] = {dc->x, dc->q, dc->attn, dc->h, dc->logits, dc->score,
                   dc->kcache, dc->vcache, dc->sin_t, dc->cos_t, dc->tp_tmp, dc->k_raw};
  for (float* b : bufs)
    if (b) cudaFree(b);
  if (dc->st) cudaFree(dc->st);
  if (dc->out_tokens) cudaFree(dc->out_tokens);
  if (dc->teacher) cudaFree(dc->teacher);
  if (dc->pf_buf) cudaFree(dc->pf_buf);
  if (dc->pf_w8_ws) cudaFree(dc->pf_w8_ws);
  if (dc->st_host) cudaFreeHost(dc->st_host);
  if (dc->io_host) cudaFreeHost(dc->io_host);
  if (dc->own_stream && dc->stream) cudaStreamDestroy(dc->stream);
  delete dc;
}

int kllm_decoder_step(kllm_decoder* dc, int32_t token_host, int32_t pos, int is_prompt,
                      int32_t* next_host) {
  if (!dc || !next_host) return KLLM_E_INVALID;
  if (pos < 0 || pos >= dc->d.seq_len) return KLLM_E_INVALID;
  StepState* hs = dc->st_host;
  hs->token = token_host;
  hs->pos = pos;
  hs->step = 0;
  hs->next = -1;
  KLLM_TRY(cudaMemcpyAsync(dc->st, hs, sizeof(StepState), cudaMemcpyHostToDevice, dc->stream));
  if (dc->use_mega) {
    // a prompt position needs no logits (llama3.cpp:738-739 returns -1): the classifier is skipped
    KLLM_TRY(dc->mega.run(1, nullptr, nullptr, -1, is_prompt ? 1 : 0));
  } else {
    KLLM_TRY(cudaGraphLaunch(dc->exec, dc->stream));
    count_launch(static_cast<uint64_t>(dc->launches_per_step));
  }
  KLLM_TRY(cudaMemcpyAsync(hs, dc->st, sizeof(StepState), cudaMemcpyDeviceToHost, dc->stream));
  KLLM_TRY(cudaStreamSynchronize(dc->stream));
  *next_host = is_prompt ? -1 : hs->next;
  return 0;
}

int kllm_decoder_prompt(kllm_decoder* dc, const int32_t* tokens_host, int32_t n_tokens, int32_t start_pos,
                        int32_t* next_host) {
  if (!dc || !tokens_host || !next_host || n_tokens <= 0 || start_pos < 0) return KLLM_E_INVALID;
  if (start_pos + n_tokens > dc->d.seq_len) return KLLM_E_INVALID;
  StepState* hs = dc->st_host;
  hs->token = tokens_host[0];
  hs->pos = start_pos;
  hs->step = 0;
  hs->next = -1;
  KLLM_TRY(cudaMemcpyAsync(dc->st, hs, sizeof(StepState), cudaMemcpyHostToDevice, dc->stream));
  std::memcpy(dc->io_host, tokens_host, sizeof(int32_t) * n_tokens);
  KLLM_TRY(cudaMemcpyAsync(dc->teacher, dc->io_host, sizeof(int32_t) * n_tokens, cudaMemcpyHostToDevice,
                           dc->stream));
  if (dc->use_mega) {
    // ONE launch for the whole prompt; only the last position runs the classifier
    KLLM_TRY(dc->mega.run(n_tokens, dc->teacher, nullptr, -1, n_tokens - 1));
  } else {
    for (int i = 0; i < n_tokens; ++i) KLLM_TRY(cudaGraphLaunch(dc->exec_tf, dc->stream));
    count_launch(static_cast<uint64_t>(dc->launches_per_step) * n_tokens);
  }
  KLLM_TRY(cudaMemcpyAsync(hs, dc->st, sizeof(StepState), cudaMemcpyDeviceToHost, dc->stream));
  KLLM_TRY(cudaStreamSynchronize(dc->stream));
  *next_host = hs->next;
  return 0;
}

}  // extern "C"

namespace {

// Batched prefill shared by kllm_decoder_prefill_tf32 (fp32 weights, kllm_gemm_tf32) and
// kllm_decoder_prefill_w8 (int8 group-64 weights, kllm_gemm_w8); the callers check the checkpoint kind.
int prefill_batched(kllm_decoder* dc, const int32_t* tokens_host, int32_t n_tokens, int32_t start_pos,
                    int32_t* next_host, bool w8) {
  constexpr int kBlock = 256;  // prompt positions per pass = the N of the tcgen05.mma (tf32)
  const kllm_decoder_desc& d = dc->d;
  const int hs = dc->head_size, q_rows = d.head_num * hs, kvd = dc->kv_dim;
  if (w8 && dc->pf_w8_ws == nullptr) {  // the GEMM's digit planes + steps for the widest input of a block
    const size_t kmax = static_cast<size_t>(std::max(std::max(d.dim, d.hidden_dim), q_rows));
    const size_t bytes = 3 * kBlock * kmax + 4 * (kmax / 64) * kBlock;
    if (cudaMalloc(&dc->pf_w8_ws, bytes) != cudaSuccess) return static_cast<int>(cudaErrorMemoryAllocation);
  }
  if (dc->pf_buf == nullptr) {
    const size_t per_row = static_cast<size_t>(3 * d.dim + 2 * q_rows + 2 * kvd + 2 * d.hidden_dim);
    if (cudaMalloc(&dc->pf_buf, per_row * kBlock * sizeof(float)) != cudaSuccess)
      return static_cast<int>(cudaErrorMemoryAllocation);
    float* p = dc->pf_buf;
    auto take = [&](size_t n) {
      float* r = p;
      p += n * kBlock;
      return r;
    };
    dc->pf_ws.x = take(d.dim), dc->pf_ws.xn = take(d.dim), dc->pf_ws.tmp = take(d.dim);
    dc->pf_ws.q = take(q_rows), dc->pf_ws.att = take(q_rows);
    dc->pf_ws.k = take(kvd), dc->pf_ws.v = take(kvd);
    dc->pf_ws.h1 = take(d.hidden_dim), dc->pf_ws.h3 = take(d.hidden_dim);
  }
  KLLM_TRY(prefill_attention_smem_opt_in(static_cast<size_t>(start_pos + n_tokens) * sizeof(float)));
  PrefillModel m{};
  m.dim = d.dim, m.hidden_dim = d.hidden_dim, m.layer_num = d.layer_num, m.head_num = d.head_num;
  m.kv_head_num = d.kv_head_num, m.vocab_size = d.vocab_size, m.seq_len = d.seq_len, m.head_size = hs;
  m.flavour = d.flavour, m.mega_layout = dc->use_mega ? 1 : 0, m.eps = flavour_eps(d.flavour);
  m.attn_split = dc->use_mega ? dc->mega.attn_vsplit() : 1;
  m.tok_emb = d.tok_emb, m.attn_norm = dc->attn_norm.data(), m.ffn_norm = dc->ffn_norm.data();
  m.wq = dc->wq.data(), m.wk = dc->wk.data(), m.wv = dc->wv.data(), m.wo = dc->wo.data();
  m.w1 = dc->w1.data(), m.w2 = dc->w2.data(), m.w3 = dc->w3.data();
  if (w8) {
    m.sq = dc->sq.data(), m.sk = dc->sk.data(), m.sv = dc->sv.data(), m.so = dc->so.data();
    m.s1 = dc->s1.data(), m.s2 = dc->s2.data(), m.s3 = dc->s3.data();
    m.w8_workspace = dc->pf_w8_ws;
  }
  m.bq = dc->bq.empty() ? nullptr : dc->bq.data();
  m.bk = dc->bk.empty() ? nullptr : dc->bk.data();
  m.bv = dc->bv.empty() ? nullptr : dc->bv.data();
  m.key_cache = dc->kcache, m.value_cache = dc->vcache, m.sin_cache = dc->sin_t, m.cos_cache = dc->cos_t;

  std::memcpy(dc->io_host, tokens_host, sizeof(int32_t) * n_tokens);
  KLLM_TRY(cudaMemcpyAsync(dc->teacher, dc->io_host, sizeof(int32_t) * n_tokens, cudaMemcpyHostToDevice, dc->stream));
  int last_rows = 0;
  for (int c0 = 0; c0 < n_tokens; c0 += kBlock) {
    const int T = std::min(kBlock, n_tokens - c0);
    KLLM_TRY(prefill_block(m, dc->pf_ws, dc->teacher + c0, T, start_pos + c0, dc->stream));
    last_rows = T;
  }
  // last prompt position only: final RMSNorm + classifier (cls_logits, llama3.cpp:722-731) and the
  // greedy id (post_processing, :733-745) through the decode path's fused GEMV and argmax
  StepState* hs_state = dc->st_host;
  hs_state->token = tokens_host[n_tokens - 1];
  hs_state->pos = start_pos + n_tokens - 1;
  hs_state->step = 0;
  hs_state->next = -1;
  KLLM_TRY(cudaMemcpyAsync(dc->st, hs_state, sizeof(StepState), cudaMemcpyHostToDevice, dc->stream));
  {
    kllm_gemv_job j{};
    j.x = dc->pf_ws.x + static_cast<size_t>(last_rows - 1) * d.dim;
    j.norm_w = d.final_norm;
    j.norm_eps = flavour_eps(d.flavour);
    j.in_dim = d.dim;
    j.group_size = d.group_size;
    j.n_seg = 1;
    j.seg[0] = {d.wcls, d.group_size ? d.scls : nullptr, nullptr, dc->logits, d.vocab_size};
    KLLM_TRY(gemv_dispatch(&j, GemvExtra{}, dc->stream));
  }
  argmax_advance_kernel<<<1, 1024, 0, dc->stream>>>(dc->logits, d.vocab_size, dc->st, nullptr, nullptr, d.seq_len);
  count_launch();
  KLLM_TRY(cudaGetLastError());
  KLLM_TRY(cudaMemcpyAsync(hs_state, dc->st, sizeof(StepState), cudaMemcpyDeviceToHost, dc->stream));
  KLLM_TRY(cudaStreamSynchronize(dc->stream));
  *next_host = hs_state->next;
  return 0;
}

}  // namespace

extern "C" {

int kllm_decoder_prefill_tf32(kllm_decoder* dc, const int32_t* tokens_host, int32_t n_tokens, int32_t start_pos,
                              int32_t* next_host) {
  if (!dc || !tokens_host || !next_host || n_tokens <= 0 || start_pos < 0) return KLLM_E_INVALID;
  const kllm_decoder_desc& d = dc->d;
  if (start_pos + n_tokens > d.seq_len) return KLLM_E_INVALID;
  if (d.group_size != 0 || d.tp_size > 1) return KLLM_E_UNSUPPORTED;  // fp32 checkpoints, one GPU
  const int q_rows = d.head_num * dc->head_size;
  if ((d.dim & 3) || (d.hidden_dim & 3) || (q_rows & 3)) return KLLM_E_UNSUPPORTED;
  return prefill_batched(dc, tokens_host, n_tokens, start_pos, next_host, false);
}

int kllm_decoder_prefill_w8(kllm_decoder* dc, const int32_t* tokens_host, int32_t n_tokens, int32_t start_pos,
                            int32_t* next_host) {
  if (!dc || !tokens_host || !next_host || n_tokens <= 0 || start_pos < 0) return KLLM_E_INVALID;
  const kllm_decoder_desc& d = dc->d;
  if (start_pos + n_tokens > d.seq_len) return KLLM_E_INVALID;
  if (d.group_size != 64 || d.tp_size > 1) return KLLM_E_UNSUPPORTED;  // int8 group-64 checkpoints, one GPU
  const int q_rows = d.head_num * dc->head_size;
  if ((d.dim % 64) || (d.hidden_dim % 64) || (q_rows % 64)) return KLLM_E_UNSUPPORTED;  // whole groups per row
  return prefill_batched(dc, tokens_host, n_tokens, start_pos, next_host, true);
}

int kllm_decoder_generate(kllm_decoder* dc, int32_t first_token, int32_t start_pos,
                          int32_t n_steps, const int32_t* teacher_host,
                          int32_t* out_tokens_host) {
  if (!dc || n_steps <= 0 || start_pos < 0) return KLLM_E_INVALID;
  if (start_pos + n_steps > dc->d.seq_len) return KLLM_E_INVALID;
  StepState* hs = dc->st_host;
  hs->token = teacher_host ? teacher_host[0] : first_token;
  hs->pos = start_pos;
  hs->step = 0;
  hs->next = -1;
  KLLM_TRY(cudaMemcpyAsync(dc->st, hs, sizeof(StepState), cudaMemcpyHostToDevice, dc->stream));
  if (teacher_host) {
    std::memcpy(dc->io_host, teacher_host, sizeof(int32_t) * n_steps);
    KLLM_TRY(cudaMemcpyAsync(dc->teacher, dc->io_host, sizeof(int32_t) * n_steps,
                             cudaMemcpyHostToDevice, dc->stream));
  }
  if (dc->use_mega) {
    KLLM_TRY(dc->mega.run(n_steps, teacher_host ? dc->teacher : nullptr));
  } else {
    cudaGraphExec_t exec = teacher_host ? dc->exec_tf : dc->exec;
    for (int i = 0; i < n_steps; ++i) KLLM_TRY(cudaGraphLaunch(exec, dc->stream));
    count_launch(static_cast<uint64_t>(dc->launches_per_step) * n_steps);
  }
  if (out_tokens_host) {
    KLLM_TRY(cudaMemcpyAsync(dc->io_host, dc->out_tokens, sizeof(int32_t) * n_steps,
                             cudaMemcpyDeviceToHost, dc->stream));
  }
  KLLM_TRY(cudaStreamSynchronize(dc->stream));
  if (out_tokens_host) std::memcpy(out_tokens_host, dc->io_host, sizeof(int32_t) * n_steps);
  return 0;
}

int kllm_decoder_profile(kllm_decoder* dc, int32_t first_token, int32_t start_pos, int32_t n_steps,
                         int32_t profiled_step, uint64_t* stamps_host, int32_t capacity,
                         int32_t* grid_out, int32_t* phases_out) {
  if (!dc || !stamps_host || !grid_out || !phases_out || n_steps <= 0) return KLLM_E_INVALID;
  if (!dc->use_mega) return KLLM_E_UNSUPPORTED;
  if (start_pos < 0 || start_pos + n_steps > dc->d.seq_len) return KLLM_E_INVALID;
  const int grid = dc->mega.grid(), phases = dc->mega.phases();
  const size_t n = static_cast<size_t>(grid) * phases * mega::kProfStamps;
  *grid_out = grid;
  *phases_out = phases;
  if (static_cast<size_t>(capacity) < n) return KLLM_E_INVALID;
  unsigned long long* d_prof = nullptr;
  KLLM_TRY(cudaMalloc(&d_prof, n * sizeof(unsigned long long)));
  cudaMemsetAsync(d_prof, 0, n * sizeof(unsigned long long), dc->stream);
  StepState* hs = dc->st_host;
  hs->token = first_token, hs->pos = start_pos, hs->step = 0, hs->next = -1;
  cudaMemcpyAsync(dc->st, hs, sizeof(StepState), cudaMemcpyHostToDevice, dc->stream);
  int rc = dc->mega.run(n_steps, nullptr, d_prof, profiled_step);
  if (rc == 0) rc = static_cast<int>(cudaStreamSynchronize(dc->stream));
  if (rc == 0)
    rc = static_cast<int>(cudaMemcpy(stamps_host, d_prof, n * sizeof(unsigned long long),
                                     cudaMemcpyDeviceToHost));
  cudaFree(d_prof);
  return rc;
}

int kllm_decoder_logits(kllm_decoder* dc, float* logits_host) {
  if (!dc || !logits_host) return KLLM_E_INVALID;
  KLLM_TRY(cudaStreamSynchronize(dc->stream));
  return static_cast<int>(cudaMemcpy(logits_host, dc->logits, sizeof(float) * dc->d.vocab_size,
                                     cudaMemcpyDeviceToHost));
}

const float* kllm_decoder_logits_device(const kllm_decoder* dc) { return dc ? dc->logits : nullptr; }

int kllm_decoder_read_kv(kllm_decoder* dc, float* key_host, float* value_host) {
  if (!dc || !key_host || !value_host) return KLLM_E_INVALID;
  KLLM_TRY(cudaStreamSynchronize(dc->stream));
  const size_t L = dc->d.layer_num, S = dc->d.seq_len, kvd = dc->kv_dim, hs = dc->head_size;
  const size_t n = L * S * kvd;
  if (!dc->use_mega) {
    KLLM_TRY(cudaMemcpy(key_host, dc->kcache, n * sizeof(float), cudaMemcpyDeviceToHost));
    return static_cast<int>(cudaMemcpy(value_host, dc->vcache, n * sizeof(float), cudaMemcpyDeviceToHost));
  }
  // persistent engine: K [L][kvh][hs/4][S][4], V [L][kvh][SP][S][hs/SP] -> reference [L][S][kv_dim]
  std::vector<float> kraw(n), vraw(n);
  KLLM_TRY(cudaMemcpy(kraw.data(), dc->kcache, n * sizeof(float), cudaMemcpyDeviceToHost));
  KLLM_TRY(cudaMemcpy(vraw.data(), dc->vcache, n * sizeof(float), cudaMemcpyDeviceToHost));
  const size_t nh = kvd / hs;
  const size_t SP = static_cast<size_t>(dc->mega.attn_vsplit()), dv = hs / SP;
  for (size_t l = 0; l < L; ++l)
    for (size_t g = 0; g < nh; ++g) {
      const float* kb = kraw.data() + (l * nh + g) * S * hs;
      const float* vb = vraw.data() + (l * nh + g) * S * hs;
      for (size_t t = 0; t < S; ++t)
        for (size_t i = 0; i < hs; ++i) {
          const size_t dst = (l * S + t) * kvd + g * hs + i;
          key_host[dst] = kb[((i >> 2) * S + t) * 4 + (i & 3)];
          value_host[dst] = vb[((i / dv) * S + t) * dv + i % dv];
        }
    }
  return 0;
}
int kllm_decoder_launches_per_step(const kllm_decoder* dc) { return dc ? dc->launches_per_step : 0; }
int kllm_decoder_classifier_rows(const kllm_decoder* dc) {
  if (!dc) return 0;
  return dc->use_mega ? dc->mega.cls_rows() : dc->d.vocab_size;
}
const char* kllm_decoder_engine(const kllm_decoder* dc) {
  if (!dc) return "";
  return dc->use_mega ? "persistent" : "graph";
}

}  // extern "C"
