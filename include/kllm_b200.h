/* kllm_b200.h -- C-ABI of the B200-native KuiperLLama decode path (libkllm_b200.so).
 *
 * This is the drop-in boundary: plain pointers, ints and an opaque stream, no C++ or torch
 * types.  Every entry point names the reference interface it replaces (paths relative to the
 * zjhellofss/KuiperLLama tree).  The C++ adapters that keep the reference's
 * `kernel::get_*_kernel(DeviceType)` registry signatures verbatim live in
 * kuiperllama_b200/kuiper/source/op/kernels/ and only translate tensor::Tensor -> pointers.
 *
 * Conventions
 *   - all data pointers are DEVICE pointers unless the parameter name ends in `_host`;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream), exactly as
 *     the reference passes `void* stream` / `CudaConfig::stream`;
 *   - functions enqueue work and return without synchronising unless documented otherwise;
 *   - return value: 0 = ok, >0 = cudaError_t from the launch, <0 = KLLM_E_* argument error
 *     (the reference CHECK-aborts instead; the C++ adapters turn non-zero into LOG(FATAL));
 *   - there is NO CPU fallback: without a CUDA device every call returns an error.
 *
 * Arithmetic contract: fp32 throughout, each kernel reproduces the reference CUDA kernel's
 * floating-point operation order (see DESIGN.md "Bit-exactness"), so results are bit-identical
 * to the reference's own CUDA path compiled for sm_100a, not merely within tolerance.
 */
#ifndef KLLM_B200_H_
#define KLLM_B200_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KLLM_OK 0
#define KLLM_E_INVALID (-1)     /* bad argument (null pointer, non-positive size, ...) */
#define KLLM_E_UNSUPPORTED (-2) /* shape outside what the kernels handle */
#define KLLM_E_STATE (-3)       /* decoder used before/after its valid life cycle */
#define KLLM_E_NODEVICE (-4)    /* no usable CUDA device */
#define KLLM_E_COMM (-5)        /* tensor-parallel transport unavailable / collective failed */

/* RoPE pairing / constants = the reference's compile-time flavour (CMakeLists.txt:16-25). */
#define KLLM_FLAVOUR_LLAMA2 0 /* interleaved pairs, theta 1e4, eps 1e-5 */
#define KLLM_FLAVOUR_LLAMA3 1 /* half-split pairs, theta 5e5, eps 1e-5 */
#define KLLM_FLAVOUR_QWEN2 2  /* half-split pairs, theta 1e6, eps 1e-6, qkv bias */

const char* kllm_version(void);
const char* kllm_error_string(int code);
/* Number of kernel launches issued through this library since load (bench.py's gpu_launches). */
uint64_t kllm_launch_count(void);

/* ---- registry-level ops ---------------------------------------------------------------
 * One per `kernel::get_*_kernel(kDeviceCUDA)` entry (kernels_interface.h:6-68).            */

/* MatmulKernel  -> matmul_kernel_cu, cuda/matmul_kernel.cu:89-109.
 * out[out_dim] = W[out_dim,in_dim] . x[in_dim], W row-major. */
int kllm_gemv_f32(const float* x, const float* w, float* out, int in_dim, int out_dim,
                  void* stream);

/* MatmulKernelQuant -> matmul_kernel_cu_qint8, cuda/matmul_kernel.cu:111-134.
 * out[p] = sum_i x[i] * scales[(p*in_dim+i)/group_size] * (float)w[p*in_dim+i]. */
int kllm_gemv_w8(const float* x, const int8_t* w, const float* scales, float* out, int in_dim,
                 int out_dim, int group_size, void* stream);

/* RMSNormKernel -> rmsnorm_kernel_cu, cuda/rmsnorm_kernel.cu:52-78 (eps is the flavour
 * constant there; here it is an argument). In-place (out == x) is allowed. */
int kllm_rmsnorm_f32(const float* x, const float* w, float* out, int n, float eps, void* stream);

/* AddKernel -> add_kernel_cu, cuda/add_kernel.cu:14-32. */
int kllm_add_f32(const float* a, const float* b, float* out, int n, void* stream);

/* SwigluKernel -> swiglu_kernel_cu, cuda/swiglu_kernel.cu:24-47: out = (x1*sigmoid(x1))*x3. */
int kllm_swiglu_f32(const float* x1, const float* x3, float* out, int n, void* stream);

/* sin_cos_cache_calc_cu, cuda/rope_kernel.cu:138-151: tables [seq_len, head_size]. */
int kllm_sincos_init(int head_size, int seq_len, int flavour, float* sin_cache, float* cos_cache,
                     void* stream);

/* RoPEKernel -> rope_kernel_cu, cuda/rope_kernel.cu:153-170. q[dim], k[kv_dim] rotated in
 * place.  `pos` by value (the reference dereferences a host int32 tensor, :157).  Unlike the
 * reference's half-split kernels (:13,:59 `idx > total_pairs`) nothing is touched out of
 * bounds. */
int kllm_rope_f32(int flavour, int dim, int kv_dim, int head_size, float* q, float* k, int pos,
                  const float* sin_cache, const float* cos_cache, void* stream);

/* MHAKernel -> mha_kernel_cu, cuda/mha_kernel.cu:112-130.  key/value cache layout
 * [layer][seq_len][kv_dim] fp32; score is the [head_num, seq_len] workspace the reference
 * also takes (left holding the softmax probabilities, as the reference leaves it). */
int kllm_mha_decode_f32(int pos, int head_num, int layer_index, int seq_len, int kv_dim,
                        int kv_mul, int head_size, float* mha_out, const float* query,
                        float* score, const float* key_cache, const float* value_cache,
                        void* stream);

/* EmbeddingKernel -> emb_kernel_cu, cuda/emb_kernel.cu:23-48.  tokens are DEVICE int32 here
 * (the reference does a blocking H2D copy of a host tensor per call, :25-29). Tokens outside
 * [0, vocab) leave their output row untouched, as the reference does. */
int kllm_embedding_f32(const int32_t* tokens, int n_tokens, const float* table, float* out,
                       int dim, int vocab, void* stream);

/* argmax_kernel_cu, cuda/argmax_kernel.cu:73-87: greedy id, lowest index on ties.
 * Result goes to *out_index (device, int64); no allocation, no synchronisation. */
int kllm_argmax_f32(const float* logits, int64_t n, int64_t* out_index, void* stream);
/* Convenience with the reference's blocking semantics: returns the index or <0 on error. */
int64_t kllm_argmax_f32_sync(const float* logits, int64_t n, void* stream);

/* ---- fused per-layer entry points -------------------------------------------------------
 * What LLama2Model::forward (llama3.cpp:147-167) calls instead of 15 launches per layer.
 * All are compositions of the ops above with identical arithmetic.                          */

typedef struct {
  const void* w;       /* fp32 or int8 [rows, in_dim] row-major */
  const float* scales; /* int8 only: fp32 [rows*in_dim/group_size] */
  const float* bias;   /* optional [rows] (Qwen2 q/k/v), added after the dot product */
  float* out;          /* [rows] */
  int rows;
} kllm_gemv_seg;

typedef struct {
  const float* x;       /* [in_dim] input activation */
  const float* norm_w;  /* optional: RMSNorm weight applied to x first (attention_rms /
                           ffn rmsnorm, llama3.cpp:600-609,687-691) */
  float norm_eps;
  float* norm_out;      /* optional: where the normalised x is also written (the reference
                           keeps it in kOutputRMSNorm) */
  int in_dim;
  int group_size;       /* 0 = fp32 weights, else int8 group size */
  int n_seg;            /* 1..3 row segments sharing x (q|k|v, or w1|w3) */
  kllm_gemv_seg seg[3];
  /* epilogue */
  const float* residual; /* optional: out[p] = residual[p] + dot (VecAdd, llama3.cpp:683,719) */
  int swiglu_pair;       /* 1: n_seg==2, seg[0]=w1, seg[1]=w3, seg[0].out = swiglu(d1, d3) */
} kllm_gemv_job;

int kllm_gemv_fused(const kllm_gemv_job* job, void* stream);

/* ---- batched prompt GEMM on the tcgen05 tensor cores (TOLERANCED: TF32 multiply, fp32 accumulate) ----
 * out[n_tokens, out_dim] = x[n_tokens, in_dim] . w[out_dim, in_dim]^T, all fp32 row-major device memory.
 * Replaces the n_tokens single-row GEMVs the reference issues for a prompt, one full forward per
 * prompt token (demo/main.cpp:18-23 -> LLama2Model::predict, llama3.cpp:147-167; MatmulLayer::forward,
 * matmul.cpp:57-80): the weight matrix is streamed once per 256 tokens instead of once per token.
 * TMA tensor-map loads (cp.async.bulk.tensor, 128-byte swizzle) feed tcgen05.mma.kind::tf32 with the
 * accumulator in TMEM.  Results agree with the fp32 GEMV to ~1e-3 relative (10-bit mantissas), NOT
 * bit for bit: the decode path never uses it.  in_dim % 4 == 0, 16-byte aligned x and w. */
int kllm_gemm_tf32(const float* x, const float* w, float* out, int n_tokens, int in_dim, int out_dim,
                   void* stream);

/* ---- batched prompt GEMM, int8 weights, on tcgen05.mma.kind::i8 (TOLERANCED: x rounded to 24-bit fixed point) ----
 * out[n_tokens, out_dim] = x[n_tokens, in_dim] . (s (.) w)[out_dim, in_dim]^T with w int8 row-major and
 * scales[(p*in_dim + i) / 64] the fp32 scale of weight (p, i) -- the int8 GEMV's formula with group_size 64
 * (kllm_gemv_w8, export.py --version 3).  Each token's 64-element groups of x become step * q, step =
 * max|x in group| * 2^-22, q = rint(x / step) as three int8 digit planes (the fast decode mode's definition,
 * KLLM_NUMERICS_FAST); the int8 x int8 products of each group are exact in int32 on the tensor cores and are
 * combined with s * step in fp32.  Only x is rounded, by at most 2^-23 of its group maximum, so results agree
 * with the exact int8 GEMV to ~1e-6 relative (tests/test_prefill_w8_gpu.py states the bound), NOT bit for bit.
 * `workspace`: caller-owned device memory of KLLM_GEMM_W8_WORKSPACE_BYTES(n_tokens, in_dim) bytes for the digit
 * planes and steps (overwritten; do not share it between calls in flight on different streams).  No
 * allocation, no synchronisation.  Limits: in_dim % 64 == 0 (else KLLM_E_UNSUPPORTED); x, w and workspace
 * 16-byte aligned, scales and out 4-byte aligned (else KLLM_E_UNSUPPORTED); any n_tokens, out_dim >= 1. */
#define KLLM_GEMM_W8_WORKSPACE_BYTES(n_tokens, in_dim) \
  (3 * (size_t)(n_tokens) * (size_t)(in_dim) + 4 * ((size_t)(in_dim) / 64) * (((size_t)(n_tokens) + 63) / 64 * 64))
int kllm_gemm_w8(const float* x, const int8_t* w, const float* scales, float* out, void* workspace, int n_tokens,
                 int in_dim, int out_dim, void* stream);

/* ---- tensor-parallel exchange --------------------------------------------------------------
 * Not in the reference (single GPU: llama3.cpp:118 pins device 0); SURVEY.md section 8e.  One
 * process per GPU; each owns a kllm_comm.  The decoder issues exactly two all-reduces per layer:
 * after o_proj (before the residual add of llama3.cpp:683-684) and after down_proj (:719).
 *   KLLM_COMM_PEER: one-shot all-reduce over NVLink peer memory (CUDA IPC), rank-ordered sum,
 *                   residual add fused; set up = create on every rank, exchange the 64-byte IPC
 *                   handles out of band, connect, barrier.
 *   KLLM_COMM_NCCL: ncclAllReduce on the decoder's stream (libnccl dlopen'ed at run time);
 *                   set up = unique_id on rank 0, broadcast the 128 bytes, create everywhere.  */
#define KLLM_COMM_PEER 0
#define KLLM_COMM_NCCL 1
typedef struct kllm_comm kllm_comm;
int kllm_comm_unique_id(unsigned char* out128);
/* max_count: largest vector (floats, multiple of 4) ever reduced = the model dim. */
int kllm_comm_create(int world, int rank, int backend, int max_count, const unsigned char* nccl_id128,
                     kllm_comm** out);
int kllm_comm_ipc_handle(kllm_comm* comm, unsigned char* out64);
/* handles: world x 64 bytes, rank-ordered (own entry ignored).  Every rank must have connected
 * (caller barrier) before the first all-reduce, and must stop reducing before any rank destroys. */
int kllm_comm_connect(kllm_comm* comm, const unsigned char* handles);
/* out = (residual ? residual : 0) + sum over ranks of `partial`, summed in rank order; all
 * device pointers, 16-byte aligned, count a multiple of 4.  `partial` is clobbered (NCCL). */
int kllm_comm_allreduce_residual(kllm_comm* comm, const float* partial, const float* residual, float* out,
                                 int count, void* stream);
/* In-place sum; signature of kllm_decoder_desc.allreduce (ctx = the kllm_comm). */
int kllm_comm_allreduce(void* comm, float* buf, int count, void* stream);
int kllm_comm_info(const kllm_comm* comm, int* world, int* rank, int* backend);
void kllm_comm_destroy(kllm_comm* comm);

/* ---- whole decoder ------------------------------------------------------------------------
 * Device-resident model: replaces Model::{init_mem,forward,predict,post_processing,embedding,
 * fill_input} (llama3.cpp:425-500,147-167,642-650,733-745,578-598; model.cpp:245-263) for the
 * per-token loop of demo/main.cpp:18-41.  Weights stay where the caller put them (device);
 * the decoder owns activations, KV cache, sin/cos tables and a captured CUDA graph.        */

typedef struct {
  int32_t dim, hidden_dim, layer_num, head_num, kv_head_num, vocab_size, seq_len;
  int32_t flavour;     /* KLLM_FLAVOUR_* */
  int32_t group_size;  /* 0 = fp32 weights; 64 = export.py --version 3 int8 */
  /* device pointers, reference checkpoint order (SURVEY.md Appendix A); per-layer arrays are
   * HOST arrays of layer_num device pointers. */
  const float* tok_emb;               /* [vocab, dim] */
  const float* const* attn_norm;      /* [L] -> [dim] */
  const float* const* ffn_norm;       /* [L] -> [dim] */
  const float* final_norm;            /* [dim] */
  const void* const* wq; const void* const* wk; const void* const* wv; const void* const* wo;
  const void* const* w1; const void* const* w2; const void* const* w3;
  const void* wcls;                   /* [vocab, dim] (== tok_emb when shared, fp32 only) */
  /* int8 only: fp32 scale blocks, same shapes / group_size */
  const float* const* sq; const float* const* sk; const float* const* sv; const float* const* so;
  const float* const* s1; const float* const* s2; const float* const* s3;
  const float* scls;
  /* Qwen2 only (may be NULL): */
  const float* const* bq; const float* const* bk; const float* const* bv;
  /* tensor parallel: this rank's shard description (tp_size 1 = single GPU).  With tp_size>1
   * wq/wk/wv/w1/w3 hold this rank's ROWS, wo/w2 this rank's input COLUMNS (repacked
   * contiguous), head_num/kv_head_num/hidden_dim above are the LOCAL counts and `dim` is the
   * full model dim.  allreduce is called after o_proj and after down_proj. */
  int32_t tp_size, tp_rank;
  int (*allreduce)(void* ctx, float* buf, int count, void* stream);
  void* allreduce_ctx;
  /* preferred over the callback when set: the decoder then uses the fused
   * all-reduce + residual add of kllm_comm_allreduce_residual */
  kllm_comm* comm;
  /* Numerics of the persistent engine.  KLLM_NUMERICS_EXACT (0, the default of a zeroed struct): every
   * reduction in the reference's order -- logits and ids bit-identical to the reference's CUDA path
   * (the verification mode).  KLLM_NUMERICS_FAST (1): free summation order where it buys speed --
   * int8 rows as fixed-point activations x int8 weights on dp4a, attention as flash-decoding (split by
   * timestep, online softmax) -- within the north-star tolerance (|dlogit| <= 1e-4, same greedy ids
   * where the top-2 margin exceeds 2e-4; tests/test_decoder_gpu.py).  Environment KLLM_MODE=exact|fast
   * overrides this field at create time. */
  int32_t numerics;
} kllm_decoder_desc;
#define KLLM_NUMERICS_EXACT 0
#define KLLM_NUMERICS_FAST 1

typedef struct kllm_decoder kllm_decoder;

/* `stream`: the cudaStream_t every launch and copy of this decoder is ordered on.  NULL = the decoder
 * creates a private non-blocking stream and device-synchronises once here, so weights uploaded on
 * any other stream before this call are complete; with a caller's stream the caller orders its
 * uploads before the first step (same stream, or an event). */
int kllm_decoder_create(const kllm_decoder_desc* desc, void* stream, kllm_decoder** out);
void kllm_decoder_destroy(kllm_decoder* dec);

/* One position through the reference-facing path with HOST buffers: copies the token id
 * host->device, runs the captured forward for `pos`, copies the greedy id device->host and
 * synchronises (predict + post_processing semantics, llama3.cpp:642-650,733-745).
 * is_prompt != 0 mirrors predict(..., is_prompt=true): the forward runs, *next_host = -1. */
int kllm_decoder_step(kllm_decoder* dec, int32_t token_host, int32_t pos, int is_prompt,
                      int32_t* next_host);

/* The whole prompt in one call: positions start_pos .. start_pos + n_tokens - 1 take tokens_host[i] as
 * input, fill the KV cache, and *next_host is the greedy id after the LAST prompt token (what
 * demo/main.cpp:18-41 obtains by calling predict() once per prompt position with is_prompt = true and
 * discarding every result but the last).  Persistent engine: one launch, and the classifier pass --
 * which the reference runs and throws away for every prompt position (llama3.cpp:642-650, 738-739) --
 * is skipped for all but the last position.  Bit-identical KV cache and next id to stepping. */
int kllm_decoder_prompt(kllm_decoder* dec, const int32_t* tokens_host, int32_t n_tokens, int32_t start_pos,
                        int32_t* next_host);
/* TOLERANCED batched prefill: the same contract as kllm_decoder_prompt, but the prompt positions go
 * through every layer together -- each projection one GEMM [n, in] x [out, in]^T on the tcgen05
 * tensor cores (TF32 multiply, fp32 accumulate, kllm_gemm_tf32), the weights streamed once per 256
 * positions instead of once per position; classifier only for the last position.  KV-cache rows and
 * logits agree with the position-by-position path to ~1e-3 relative, NOT bit for bit (TF32 keeps 10
 * mantissa bits).  fp32 checkpoints on one GPU; KLLM_E_UNSUPPORTED otherwise (use kllm_decoder_prompt). */
int kllm_decoder_prefill_tf32(kllm_decoder* dec, const int32_t* tokens_host, int32_t n_tokens, int32_t start_pos,
                              int32_t* next_host);
/* TOLERANCED batched prefill for int8 checkpoints: the contract of kllm_decoder_prefill_tf32, with every
 * projection one kllm_gemm_w8 (int8 weights x 24-bit fixed-point activations, exact integer products on the
 * tcgen05 kind::i8 tensor cores) and the last position's classifier through the int8 GEMV.  KV-cache rows and
 * logits agree with the position-by-position path within the north-star tolerance (|dlogit| <= 1e-4,
 * tests/test_prefill_w8_gpu.py), NOT bit for bit.  group_size 64 on one GPU with dim, hidden_dim and
 * head_num * head_size multiples of 64; KLLM_E_UNSUPPORTED otherwise (fp32: kllm_decoder_prefill_tf32). */
int kllm_decoder_prefill_w8(kllm_decoder* dec, const int32_t* tokens_host, int32_t n_tokens, int32_t start_pos,
                            int32_t* next_host);
/* Device-resident greedy loop: positions start_pos .. start_pos+n_steps-1, each step feeding
 * the previous argmax back without leaving the GPU; ids copied to out_tokens_host at the end
 * (one synchronisation).  teacher_host (optional, n_steps ids) forces the inputs instead. */
int kllm_decoder_generate(kllm_decoder* dec, int32_t first_token, int32_t start_pos,
                          int32_t n_steps, const int32_t* teacher_host,
                          int32_t* out_tokens_host);

/* Blocking copies for tests: logits of the last step [vocab]; the KV cache in the REFERENCE
 * layout [layer][seq_len][kv_dim] (llama3.cpp:469-475) whatever the engine keeps internally. */
int kllm_decoder_logits(kllm_decoder* dec, float* logits_host);
/* Device pointer to the same logits [vocab] (what the reference keeps in
 * ModelBufferType::kForwardOutput, llama3.cpp:498-506); valid until the decoder is destroyed,
 * contents ordered after the last step on the decoder's stream. */
const float* kllm_decoder_logits_device(const kllm_decoder* dec);
int kllm_decoder_read_kv(kllm_decoder* dec, float* key_host, float* value_host);
/* Kernel launches one decode step issues (graph nodes; 1 for the persistent engine). */
int kllm_decoder_launches_per_step(const kllm_decoder* dec);
/* Classifier rows THIS rank streams per token: vocab_size, or vocab_size / tp_size when the
 * tensor-parallel persistent engine shards the classifier by vocabulary (cls_logits,
 * llama3.cpp:722-731, computed once across the ranks instead of once per rank).  That needs a
 * kllm_comm created with max_count >= max(dim, vocab_size / tp_size): the ranks publish their
 * logits rows through the same tagged exchange area as the o_proj / down_proj partials. */
int kllm_decoder_classifier_rows(const kllm_decoder* dec);
/* "persistent": one cooperative megakernel launch runs whole positions with a TMA-fed weight
 * ring; "graph": CUDA-graph chain of fused launches (shapes the ring does not handle, tensor
 * parallel).  Environment KLLM_ENGINE=graph|persistent forces a choice at create time. */
const char* kllm_decoder_engine(const kllm_decoder* dec);
/* Persistent engine only: run n_steps positions and record, for step `profiled_step`, sixteen
 * stamps per CTA per schedule phase into stamps_host[grid][phases][16] (capacity in uint64
 * elements).  Globaltimer ns: [0] phase entered, [1] input vector staged (+normalised), [2] last
 * ring stage consumed, [3] grid barrier passed, [10] input vector polled (before the norm).
 * SM cycles of warp 0: [4] addend prefetch, [5] dot products, [6] reductions, [7] epilogues,
 * [8] waiting for ring stages, [9] rows of a stage.  Measurement aid (profiles/). */
int kllm_decoder_profile(kllm_decoder* dec, int32_t first_token, int32_t start_pos,
                         int32_t n_steps, int32_t profiled_step, uint64_t* stamps_host,
                         int32_t capacity, int32_t* grid_out, int32_t* phases_out);

#ifdef __cplusplus
}
#endif
#endif /* KLLM_B200_H_ */
