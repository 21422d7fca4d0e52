/*
 * b200awq.h — C ABI of the B200-native W4A16 (AWQ v2 layout) quantized-linear path.
 *
 * This is the drop-in boundary: the two launchers below are what the reference's
 * extension entry points bind to,
 *
 *   gemv_forward_cuda_new(in_feats, kernel, scaling_factors, zeros, m, n, k, group_size)
 *       reference: awq/kernels/csrc/quantization_new/gemv/gemv_cuda.h:4-12,
 *                  host code gemv_cuda.cu:245-338, exported at csrc/pybind.cpp:23
 *   gemm_forward_cuda_new(in_feats, kernel, scales, zeros)
 *       reference: awq/kernels/csrc/quantization_new/gemm/gemm_cuda.h:3,
 *                  host code gemm_cuda.cu:1126-1236, exported at csrc/pybind.cpp:22
 *
 * called from awq/quantize/qmodule.py:207,218 (WQLinear.forward) and
 * tinychat/modules/fused_mlp.py:40,51,65,72.
 *
 * Conventions: plain pointers and sizes, no torch types.  All pointers are DEVICE
 * pointers.  Inputs are borrowed for the duration of the (asynchronous) launch; nothing
 * is retained, nothing is allocated, the calling thread is never synchronised with the
 * device.  Work is enqueued on `stream` (a cudaStream_t passed as void*; NULL = legacy
 * default stream).  Return value: 0 on success, a negative B200AWQ_ERR_* for rejected
 * arguments (nothing was launched), or a positive cudaError_t if the launch failed.
 *
 * Tensor layouts (exactly the reference's WQLinear buffers, awq/quantize/qmodule.py:98-137):
 *   x        [m, k]            fp16 / bf16, row-major, 16-byte aligned
 *   qweight  [n/4, k]          int16, the interleaved 4-bit packing of pack_intweight
 *                              (qmodule.py:26-65), 16-byte aligned
 *   scales   [>= k/group, n]   same dtype as x; rows beyond k/group are padding
 *   szeros   [>= k/group, n]   same dtype as x  (= -scale * zero_point, qmodule.py:194-196)
 *   y        [m, n]            same dtype as x, row-major
 * Semantics: y[i,j] = sum_k x[i,k] * rn_T( q[j,k] * scales[k/group, j] + szeros[k/group, j] )
 * with q the unsigned nibble 0..15, accumulated in fp32, rounded once to T.
 */
#ifndef B200AWQ_H_
#define B200AWQ_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200AWQ_DTYPE_F16 0
#define B200AWQ_DTYPE_BF16 1

#define B200AWQ_OK 0
#define B200AWQ_ERR_SHAPE (-1)     /* n % 8 (gemv) / n % 128 (gemm), k % 128, m out of range */
#define B200AWQ_ERR_GROUP (-2)     /* group_size != 128 (reference: gemv_cuda.cu:289,332-335) */
#define B200AWQ_ERR_ALIGN (-3)     /* a pointer is NULL or not 16-byte aligned */
#define B200AWQ_ERR_DTYPE (-4)     /* dtype is not F16 / BF16 (reference: dispatch_utils.cuh:7-18) */
#define B200AWQ_ERR_BATCH (-5)     /* gemv with m outside 1..7 (reference: gemv_cuda.cu:291-330) */
#define B200AWQ_ERR_WORKSPACE (-6) /* workspace smaller than b200awq_w4a16_gemm_workspace_bytes */
#define B200AWQ_ERR_DRIVER (-7)    /* CUDA driver entry point for TMA descriptors unavailable */
#define B200AWQ_ERR_DEVICE (-8)    /* current device is not compute capability 10.x */
#define B200AWQ_ERR_PEERS (-9)     /* bad peer description (world, rank, capacities, null buffers) */

/* Decode path: 1 <= m <= 7 (the reference's GEMV envelope).  n % 8 == 0, k % 128 == 0,
 * group_size == 128. */
int b200awq_w4a16_gemv(const void* x, const void* qweight, const void* scales, const void* szeros,
                       void* y, int m, int n, int k, int group_size, int dtype, void* stream);

/* Prefill / batched path: any m >= 1.  n % 128 == 0, k % 128 == 0, group 128 (the
 * reference GEMM hard-codes G = 128, gemm_cuda.cu:1157).  `workspace` may be NULL when
 * b200awq_w4a16_gemm_workspace_bytes(m, n, k) == 0. */
int b200awq_w4a16_gemm(const void* x, const void* qweight, const void* scales, const void* szeros,
                       void* y, int m, int n, int k, int group_size, int dtype,
                       void* workspace, size_t workspace_bytes, void* stream);

size_t b200awq_w4a16_gemm_workspace_bytes(int m, int n, int k);

/* Row-parallel tensor parallelism (new work, SURVEY.md §8e; the reference has no multi-GPU path): the decode
 * GEMV of THIS rank's k-slice fused with the sum all-reduce of the [m, n] partial outputs over NVLink peer
 * memory, in one kernel.  Every rank calls it with its own shard and the same (m, n); on return (stream order)
 * y holds the full sum on every rank, bit-identical across ranks.
 *   data[r]   rank r's exchange buffer as mapped in this process (symmetric / peer-mapped allocation):
 *             8-byte words {fp32 partial, epoch}, >= 2 * world * cap_words of them, ZERO before the first call
 *   epoch     this rank's private counters (device memory, uint32, n_max / 8 elements, ZERO before first use)
 *   n_max     widest layer (out_features) the buffers are sized for, a multiple of 8
 *   cap_words words per (parity, source rank) region = tok_cap * n_max for some tok_cap >= m; a word's slot is
 *             channel * tok_cap + token and its epoch counter is the channel's row block, so layers of
 *             DIFFERENT n (<= n_max) may share one set of buffers.
 *   1 <= m <= 8, world <= 8.  n > n_max or m > cap_words / n_max is rejected with B200AWQ_ERR_PEERS.  All ranks
 *   must issue the same sequence of calls on these buffers.  Safe under CUDA-graph capture / replay (no
 *   host-side state).  A rank whose peer delivers nothing for 10 s gives up: its outputs of that call are NaN and
 *   every later exchange of the process returns NaN at once (the kernel never spins for ever). */
typedef struct b200awq_peers {
  void* data[8];
  void* epoch;
  int rank, world;
  int cap_words;
  int n_max;
} b200awq_peers;

int b200awq_w4a16_gemv_allreduce(const void* x, const void* qweight, const void* scales, const void* szeros,
                                 void* y, int m, int n, int k, int group_size, int dtype,
                                 const b200awq_peers* peers, void* stream);

/* Front half of the gated MLP (SURVEY.md §8f-1): y = silu(x Wgate~^T) * (x Wup~^T), i.e. what
 * QuantLlamaMLP.our_llama_mlp computes with two engine calls, F.silu and a multiply
 *   reference: tinychat/modules/fused_mlp.py:36-83 (both branches use the zeros tensor they are GIVEN; the GEMM
 *   branch's `scaled_zeros - 8 * scales` is the caller's business).
 * Same tensor layouts as b200awq_w4a16_gemv / gemm for each weight set; y is [m, n].  Roundings are the reference's:
 * gate and up products rounded to T, silu (fp32) rounded to T, product rounded to T.
 *   m == 1, fp16: ONE kernel -- x read once, the two weight streams share one shared-memory ring, one [1, n] write
 *                 (no workspace needed).
 *   otherwise:    the two products through the GEMV / GEMM path into `workspace` (>= b200awq_w4a16_mlp_front_workspace_bytes
 *                 = 2 * m * n * 2 bytes, 16-byte aligned), then one elementwise kernel.  n % 128 == 0 for m >= 8. */
int b200awq_w4a16_mlp_front(const void* x, const void* gate_qweight, const void* gate_scales, const void* gate_szeros,
                            const void* up_qweight, const void* up_scales, const void* up_szeros, void* y, int m, int n, int k,
                            int group_size, int dtype, void* workspace, size_t workspace_bytes, void* stream);
size_t b200awq_w4a16_mlp_front_workspace_bytes(int m, int n, int k);

/* RMSNorm of the decoder layers around the quantised linears (SURVEY.md §8f-2): y[i, :] = x[i, :] *
 * rsqrt(mean(x[i, :]^2) + eps) * gamma, statistics in fp32, one rounding to the element type (fp16 results are
 * clamped to +-(65504 - 1000) like the reference).  Replaces layernorm_forward_cuda(input, gamma, out, eps)
 *   reference: awq/kernels/csrc/layernorm/layernorm.cu:38-64 (kernel), :111-131 (host), csrc/pybind.cpp:17.
 * x, y: [m, n] row-major, gamma: [n]; any n >= 1 (16-byte aligned pointers and n % 8 == 0 take the one-pass
 * kernel).  m == 0 is a no-op. */
int b200awq_rmsnorm(const void* x, const void* gamma, void* y, int m, int n, float eps, int dtype, void* stream);

/* Decode-step attention over tinychat's KV-cache layout (SURVEY.md §8f-3).  Replaces
 *   single_query_attention(q, k, v, k_cache, v_cache, length_per_sample, alibi_slopes, timestep, rotary_embedding_dim,
 *                          rotary_base, rotary_scale, neox_rotary_style)
 *   reference: awq/kernels/csrc/attention/ft_attention.cpp:112-184, exported at csrc/pybind.cpp:24-27, called from
 *              tinychat/modules/fused_attn.py:308-321.
 * q [batch, heads, head_dim], k / v [batch, kv_heads, head_dim] with their own batch strides in ELEMENTS (they are
 * usually views into the fused QKV output; the reference applies q's stride to all three, template.hpp:967-969), head
 * stride head_dim, unit element stride; k_cache [batch, kv_heads, head_dim / 8,
 * max_len, 8], v_cache [batch, kv_heads, max_len, head_dim], out [batch, heads, head_dim] contiguous.  The current
 * step's q and k are rotated at position t = length_per_sample ? length_per_sample[b] : timestep (angle t * scale /
 * base^(2i / rotary_dim); neox != 0 pairs (i, i + rotary_dim / 2), else (2i, 2i + 1)) and rounded to the element type;
 * k and v are stored at cache slot t % max_len; out = softmax(q K^T / sqrt(head_dim)) V over the last min(t + 1,
 * max_len) positions.  G = heads / kv_heads is any integer from 1 to 128 (query head h reads KV head h / G).
 * head_dim: a multiple of 8 up to 256 for G <= 8, a multiple of 16 up to 256 for G > 8 (every head dim the reference
 * accepts); other shapes return B200AWQ_ERR_SHAPE.
 * `workspace`: >= b200awq_single_query_attention_workspace_bytes(...) bytes of device memory, ZERO before the first
 * use, then owned by the kernels (they leave it zero where it matters); one workspace per stream.  ALiBi is not
 * supported (the reference's alibi_slopes argument must be None). */
int b200awq_single_query_attention(const void* q, const void* k, const void* v, void* k_cache, void* v_cache, void* out,
                                   const int* length_per_sample, int batch, int heads, int kv_heads, int head_dim,
                                   int max_len, int timestep, long long q_batch_stride, long long k_batch_stride,
                                   long long v_batch_stride, int rotary_dim, float rotary_base,
                                   float rotary_scale, int neox, int dtype, void* workspace, size_t workspace_bytes,
                                   void* stream);
size_t b200awq_single_query_attention_workspace_bytes(int batch, int heads, int kv_heads, int head_dim, int max_len);

/* RoPE with explicit angles over a strided [s, b, h, d] tensor (prefill).  Replaces
 *   fused_rope_with_pos_forward_func(input, freqs, transpose_output_memory)
 *   reference: awq/kernels/csrc/rope_new/fused_rope_with_pos.cu:33-75,243-285, csrc/pybind.cpp:28, called from
 *              tinychat/modules/fused_attn.py:253-254.
 * y[s, b, h, i] = x[i] cos(f_i) + rot(x)[i] sin(f_i) for i < d2 with f_i = freqs[(b * S + s) * d2 + i] (fp32) and
 * rot(x)[i] = -x[i + d2 / 2] for i < d2 / 2, x[i - d2 / 2] otherwise; elements i >= d2 are copied.  Strides in ELEMENTS
 * for s, b, h, d of the input and of the output. */
int b200awq_rope_with_pos(const void* x, const float* freqs, void* y, int s, int b, int h, int d, int d2,
                          const long long in_strides[4], const long long out_strides[4], int dtype, void* stream);

/* In-place NeoX-style RoPE on query and key from a table of cosines and sines (the HF-attention branch).  Replaces
 *   rotary_embedding_neox(positions, query, key, head_size, cos_sin_cache)
 *   reference: awq/kernels/csrc/position_embedding/pos_encoding_kernels.cu:13-88, csrc/pybind.cpp:24, called from
 *              tinychat/modules/fused_attn.py:61-79 (QuantLlamaRotaryEmbedding, table built at :43-59).
 * For every token t and head: with p = positions[t] (int64) and row = cos_sin_cache[p] ([rot_dim] of T: rot_dim / 2
 * cosines, then rot_dim / 2 sines), the pairs (x, y) = (head[r], head[rot_dim / 2 + r]), r < rot_dim / 2, become
 * (x cos_r - y sin_r, y cos_r + x sin_r); elements beyond rot_dim are untouched.  Products in fp32, one rounding to T
 * (the reference multiplies and adds in T: <= 2 ulp apart).  query [tokens, q_heads, head_size] and key
 * [tokens, k_heads, head_size] with token strides in ELEMENTS; the reference rotates key with query's head count
 * (pos_encoding_kernels.cu:61,64 -- equal for the models that take this branch), here each tensor has its own;
 * key may be NULL with k_heads == 0.  positions are not range-checked (as in the reference). */
int b200awq_rotary_embedding_neox(const long long* positions, void* query, void* key, const void* cos_sin_cache, int tokens,
                                  int q_heads, int k_heads, int head_size, int rot_dim, long long q_token_stride,
                                  long long k_token_stride, int dtype, void* stream);

/* Names used by BASELINE.json's north_star; identical to the two launchers above. */
int gemv_forward_4bit(const void* x, const void* qweight, const void* scales, const void* szeros,
                      void* y, int m, int n, int k, int group_size, int dtype, void* stream);
int gemm_forward_4bit(const void* x, const void* qweight, const void* scales, const void* szeros,
                      void* y, int m, int n, int k, int group_size, int dtype,
                      void* workspace, size_t workspace_bytes, void* stream);

/* Programmatic dependent launch between consecutive launches of this library on one
 * stream (weights of launch i+1 are prefetched while launch i drains).  Default on;
 * B200AWQ_PDL=0 in the environment or b200awq_set_pdl(0) turns it off.  Returns the
 * previous setting. */
int b200awq_set_pdl(int enable);

/* The library reads its B200AWQ_* environment knobs once, at the first launch.  Tuning / benchmarking tools that
 * change the environment inside one process call this to have them read again (thread-safe). */
void b200awq_reload_config(void);

/* Number of kernels this library has launched since load (monotonic, per process). */
unsigned long long b200awq_launch_count(void);

/* Human-readable text for a return value of the functions above. */
const char* b200awq_strerror(int code);

/* "b200awq <version> sm_100a" */
const char* b200awq_version(void);

#ifdef __cplusplus
}
#endif
#endif /* B200AWQ_H_ */
