// Decode-step attention and rotary embedding around the W4A16 linears (SURVEY.md §8f-3).
//
//  * single-query attention with the KV-cache layout tinychat's callers fix
//      k_cache [B, Hkv, D / 8, L, 8]   v_cache [B, Hkv, L, D]       (tinychat/modules/fused_attn.py:195-223)
//    replaces `single_query_attention` (awq/kernels/csrc/attention/ft_attention.cpp:112-184 ->
//    decoder_masked_multihead_attention_template.hpp:880-1500, FasterTransformer's masked MHA): per (batch, head)
//      tlength = length_per_sample ? length_per_sample[b] : timestep                        (:975-978)
//      q, k of the current step are rotated at position tlength (RoPE, angle = tlength * scale / base^(2i / rot_dim),
//      utils.h:1282-1287; neox style pairs (i, i + rot_dim / 2), else (2i, 2i + 1)) and ROUNDED to T        (:1080-1135)
//      k, v are written to the cache at slot tlength % L                                   (:1148-1175, :1424-1440)
//      out = softmax(q . K^T / sqrt(D)) V over positions max(0, tlength + 1 - L) .. tlength  (:1177-1500), fp32 math
//    ALiBi slopes and fp32 tensors are not supported here (Llama-family callers pass None / fp16, bf16).
//    B200 design: the G = H / Hkv query heads that share a KV head are served by ONE CTA (the KV bytes are read once),
//    and long contexts are SPLIT over CTAs (flash-decoding): every CTA writes (max, sum, unnormalised output) of its
//    chunk to the workspace, the last one to arrive combines.  Two kernels share the current-step prologue (rotation,
//    rounding, cache write) and that epilogue:
//      G <= 8 (any head_dim that is a multiple of 8 up to 256): CUDA cores, fp32 FMAs, 16-byte loads (K coalesces over
//        positions, V over channels); about G flop per KV byte, well under the fp32 rate at these G.
//      9 <= G <= 128 (head_dim a multiple of 16 up to 256; Qwen2, Llama-3.2-3B, Falcon, multi-query): mma.sync m16n8k16
//        with fp32 accumulators, the heads as the M dimension (tiles of 16), an online softmax per head row, P rounded to
//        T as the A operand of P.V.  K and V go from HBM straight into B fragments: the channel order of Q.K^T and the
//        channel order of the output are permuted so that each lane's 16-byte loads ARE its fragments (Q is stored in
//        shared memory in the matching order and read with ldmatrix).
//    HBM-bound: algorithmic bytes = 2 * n_pos * D * sizeof(T) per KV head.
//  * fused_rope_with_pos_forward_func (awq/kernels/csrc/rope_new/fused_rope_with_pos.cu:33-75,243-285): RoPE over a
//    strided [s, b, h, d] tensor with per-(s, b) angles `freqs`, fp32 math, one rounding.
#include <algorithm>
#include <cfloat>

#include "w4_common.cuh"
#include "w4a16_kernels.h"

namespace b200awq {
namespace {

template <typename T>
__device__ __forceinline__ float t2f(T v) {
  if constexpr (TypeTraits<T>::kIsBf16) return __bfloat162float(v);
  else return __half2float(v);
}
template <typename T>
__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 p;
    if constexpr (TypeTraits<T>::kIsBf16) p = __bfloat1622float2(u32_as_b2(w[i]));
    else p = __half22float2(u32_as_h2(w[i]));
    f[2 * i] = p.x, f[2 * i + 1] = p.y;
  }
}

constexpr int kAttThreads = 256;
constexpr int kAttMaxG = 8;      // query heads per KV head on the CUDA-core kernel
constexpr int kAttTcMaxG = 128;  // ... on the tensor-core kernel
constexpr int kAttMaxD = 256;  // head dimension
constexpr int kAttCounters = 4096;  // batch * kv_heads the workspace's counter block is sized for

struct AttArgs {
  const void* q;
  const void* k;
  const void* v;
  void* k_cache;
  void* v_cache;
  void* out;
  const int* length_per_sample;
  float* ws;            // [B][Hkv][splits][G][D + 2] partials (after the counters)
  unsigned int* count;  // [B][Hkv] arrival counters at the START of the workspace (zero between launches)
  long long q_stride, k_stride, v_stride;  // elements between batches of q / k / v
  int B, H, Hkv, D, L, timestep, rot_dim, neox, splits, chunk;
  float base, scale, inv_sqrt_d;
};

// rotate (x, y) by the angle of pair `pair_idx` at position t
__device__ __forceinline__ void rope_pair(float& x, float& y, int pair_idx, int rot_dim, int t, float base, float scale) {
  const float ang = ((float)t * scale) / powf(base, (float)(2 * pair_idx) / (float)rot_dim);
  float s, c;
  sincosf(ang, &s, &c);
  const float rx = c * x - s * y, ry = c * y + s * x;
  x = rx, y = ry;
}

// The current step, shared by both kernels.  q of the G heads of KV head `kvh` is rotated at position tlength and
// rounded to T like the reference; store_q(g, channel, value) puts it where the kernel wants it.  The CTA whose chunk
// holds the current position also rotates k, rounds it and writes k and v to cache slot tlength % L.
// Pair slot j of a head: neox style -> elements (j, j + rot_dim / 2) for j < rot_dim / 2, angle index j; interleaved ->
// elements (2 j, 2 j + 1), angle index j while 2 j < rot_dim; the remaining elements are copied.
template <typename T, typename StoreQ>
__device__ __forceinline__ void att_current_step(const AttArgs& a, int G, int b, int kvh, int tlength, bool has_current,
                                                 StoreQ&& store_q) {
  const int D = a.D, L = a.L, tid = threadIdx.x;
  const T* q = static_cast<const T*>(a.q) + (size_t)b * a.q_stride;
  const T* kin = static_cast<const T*>(a.k) + (size_t)b * a.k_stride;
  const T* vin = static_cast<const T*>(a.v) + (size_t)b * a.v_stride;
  T* kc = static_cast<T*>(a.k_cache) + (size_t)(b * a.Hkv + kvh) * L * D;
  T* vc = static_cast<T*>(a.v_cache) + (size_t)(b * a.Hkv + kvh) * L * D;
  const int half_rot = a.rot_dim >> 1;
  for (int i = tid; i < (G + 1) * (D / 2); i += kAttThreads) {
    const int g = i / (D / 2), j = i % (D / 2);            // g == G: the key
    if (g == G && !has_current) continue;
    const T* src = g < G ? q + (size_t)(kvh * G + g) * D : kin + (size_t)kvh * D;
    int i0, i1;
    bool rot;
    if (a.neox) {
      rot = j < half_rot;
      i0 = rot ? j : a.rot_dim + 2 * (j - half_rot);
      i1 = rot ? j + half_rot : i0 + 1;
    } else {
      rot = 2 * j < a.rot_dim;
      i0 = 2 * j, i1 = 2 * j + 1;
    }
    float x = t2f<T>(src[i0]), y = t2f<T>(src[i1]);
    if (rot) rope_pair(x, y, j, a.rot_dim, tlength, a.base, a.scale);
    const T xr = from_float<T>(x), yr = from_float<T>(y);
    if (g < G) {
      store_q(g, i0, xr), store_q(g, i1, yr);
    } else {                                               // k -> cache [D / 8][L][8] at slot tlength % L
      const int slot = tlength % L;
      kc[((size_t)(i0 >> 3) * L + slot) * 8 + (i0 & 7)] = xr;
      kc[((size_t)(i1 >> 3) * L + slot) * 8 + (i1 & 7)] = yr;
    }
  }
  if (has_current)
    for (int i = tid; i < D; i += kAttThreads) vc[(size_t)(tlength % L) * D + i] = vin[(size_t)kvh * D + i];
}

// The end of both kernels: value(i) is the unnormalised output of head i / D, channel i % D of this CTA's chunk,
// smax[g] / ssum[g] the max and the sum of exp(logit - max) of head g over the chunk.  One split: out = value / sum.
// Several: the CTA writes (value, max, sum) per head to its workspace slot [G][D + 2]; the last CTA of this
// (batch, KV head) to arrive combines all slots and resets the arrival counter for the next launch.
template <typename T, typename Value>
__device__ __forceinline__ void att_finish(const AttArgs& a, int G, int b, int kvh, int split, const float* smax,
                                           const float* ssum, Value&& value) {
  const int D = a.D, tid = threadIdx.x;
  float* part = a.ws + ((size_t)(b * a.Hkv + kvh) * a.splits + split) * G * (D + 2);
  T* out = static_cast<T*>(a.out) + ((size_t)b * a.H + (size_t)kvh * G) * D;
  for (int i = tid; i < G * D; i += kAttThreads) {
    const float s = value(i);
    if (a.splits == 1) out[i] = from_float<T>(s / ssum[i / D]);
    else part[(i / D) * (D + 2) + (i % D)] = s;
  }
  if (a.splits == 1) return;
  for (int g = tid; g < G; g += kAttThreads) part[g * (D + 2) + D] = smax[g], part[g * (D + 2) + D + 1] = ssum[g];
  __threadfence();
  __syncthreads();
  __shared__ unsigned int s_last;
  if (tid == 0) s_last = atomicAdd(&a.count[b * a.Hkv + kvh], 1u) == (unsigned)a.splits - 1 ? 1u : 0u;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  const float* all = a.ws + (size_t)(b * a.Hkv + kvh) * a.splits * G * (D + 2);
  for (int i = tid; i < G * D; i += kAttThreads) {
    const int g = i / D, d = i % D;
    float M = -FLT_MAX;
    for (int s = 0; s < a.splits; ++s) M = fmaxf(M, all[((size_t)s * G + g) * (D + 2) + D]);
    float num = 0.f, den = 0.f;
    for (int s = 0; s < a.splits; ++s) {
      const float* ps = all + ((size_t)s * G + g) * (D + 2);
      const float w = __expf(ps[D] - M);
      num = fmaf(w, ps[d], num), den = fmaf(w, ps[D + 1], den);
    }
    out[i] = from_float<T>(num / den);
  }
  if (tid == 0) a.count[b * a.Hkv + kvh] = 0u;  // ready for the next launch (graph replay included)
}

// resident CTAs per SM the register budget aims at (the accumulators grow with G); bf16 at G = 4 needs a few registers
// more than the 80 of three CTAs per SM and would spill there
template <typename T, int G>
constexpr int att_min_blocks() { return G <= 2 ? 4 : G <= 4 && !(TypeTraits<T>::kIsBf16 && G == 4) ? 3 : 2; }

template <typename T, int G>
__global__ void __launch_bounds__(kAttThreads, att_min_blocks<T, G>()) single_query_attention_kernel(const AttArgs a) {
  extern __shared__ __align__(16) float att_smem[];
  const int D = a.D, L = a.L;
  float* qs = att_smem;                 // [G][D] rotated, rounded queries
  float* red = qs + G * D;              // [8 warps][G] / reduction scratch (>= 16 * G * 8 for the PV reduction: below)
  float* sc = red + kAttThreads / 32 * G + 2 * G;  // [G][chunk] logits -> probabilities
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int split = blockIdx.x, kvh = blockIdx.y, b = blockIdx.z;
  T* kc = static_cast<T*>(a.k_cache) + (size_t)(b * a.Hkv + kvh) * L * D;
  T* vc = static_cast<T*>(a.v_cache) + (size_t)(b * a.Hkv + kvh) * L * D;
  pdl_launch_dependents();
  pdl_wait_prior_grid();
  const int tlength = a.length_per_sample ? a.length_per_sample[b] : a.timestep;
  const int first = max(0, tlength + 1 - L);
  const int npos = tlength + 1 - first;                   // positions attended to, the current one last
  const int p0 = first + split * a.chunk, p1 = min(first + npos, p0 + a.chunk);
  const bool has_current = p0 <= tlength && tlength < p0 + a.chunk;  // this CTA's chunk holds the current step

  // ---- current step: rotate q (every CTA) and k (the CTA that owns the current step), round to T like the reference
  att_current_step<T>(a, G, b, kvh, tlength, has_current, [&](int g, int c, T x) { qs[g * D + c] = t2f<T>(x); });
  __syncthreads();  // qs complete; this CTA's own cache writes are visible to its own reads below

  // ---- logits of this chunk: lane = position (K coalesces over positions), all G heads against one load of K
  float mx[G];
#pragma unroll
  for (int g = 0; g < G; ++g) mx[g] = -FLT_MAX;
  const int nch = D >> 3;
  for (int p = p0 + tid; p < p1; p += kAttThreads) {
    const int slot = p % L;
    float acc[G];
#pragma unroll
    for (int g = 0; g < G; ++g) acc[g] = 0.f;
    for (int c0 = 0; c0 < nch; c0 += 4) {  // four 16-byte loads in flight per position; the tail is guarded
      uint4 kv4[4];
#pragma unroll
      for (int j = 0; j < 4; ++j)
        kv4[j] = c0 + j < nch ? *reinterpret_cast<const uint4*>(kc + ((size_t)(c0 + j) * L + slot) * 8) : make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (c0 + j >= nch) break;
        const int c = c0 + j;
        float kf[8];
        unpack8<T>(kv4[j], kf);
#pragma unroll
        for (int g = 0; g < G; ++g) {
          const float4 qa = *reinterpret_cast<const float4*>(qs + g * D + c * 8);
          const float4 qb = *reinterpret_cast<const float4*>(qs + g * D + c * 8 + 4);
          acc[g] = fmaf(qa.x, kf[0], acc[g]), acc[g] = fmaf(qa.y, kf[1], acc[g]);
          acc[g] = fmaf(qa.z, kf[2], acc[g]), acc[g] = fmaf(qa.w, kf[3], acc[g]);
          acc[g] = fmaf(qb.x, kf[4], acc[g]), acc[g] = fmaf(qb.y, kf[5], acc[g]);
          acc[g] = fmaf(qb.z, kf[6], acc[g]), acc[g] = fmaf(qb.w, kf[7], acc[g]);
        }
      }
    }
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const float s = acc[g] * a.inv_sqrt_d;
      sc[g * a.chunk + (p - p0)] = s;
      mx[g] = fmaxf(mx[g], s);
    }
  }
  // block max per head
#pragma unroll
  for (int g = 0; g < G; ++g) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx[g] = fmaxf(mx[g], __shfl_xor_sync(0xffffffffu, mx[g], o));
    if (lane == 0) red[warp * G + g] = mx[g];
  }
  __syncthreads();
  float* stat = red + kAttThreads / 32 * G;  // [G] max, [G] sum
  if (tid < G) {
    float m = -FLT_MAX;
    for (int w = 0; w < kAttThreads / 32; ++w) m = fmaxf(m, red[w * G + tid]);
    stat[tid] = m;
  }
  __syncthreads();
  float sum[G];
#pragma unroll
  for (int g = 0; g < G; ++g) sum[g] = 0.f;
  for (int i = tid; i < p1 - p0; i += kAttThreads) {
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const float e = __expf(sc[g * a.chunk + i] - stat[g]);
      sc[g * a.chunk + i] = e;
      sum[g] += e;
    }
  }
  __syncthreads();  // stat[max] consumed by everybody; red reusable
#pragma unroll
  for (int g = 0; g < G; ++g) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum[g] += __shfl_xor_sync(0xffffffffu, sum[g], o);
    if (lane == 0) red[warp * G + g] = sum[g];
  }
  __syncthreads();
  if (tid < G) {
    float s = 0.f;
    for (int w = 0; w < kAttThreads / 32; ++w) s += red[w * G + tid];
    stat[G + tid] = s;
  }
  __syncthreads();

  // ---- probabilities x V: thread = (row r of 256 / (D / 8) position rows, 8 channels dc); V coalesces over channels.
  // When D / 8 does not divide 256 the last 256 % (D / 8) threads hold no row.
  const int tpr = D >> 3, rows = kAttThreads / tpr, r = tid / tpr, dc = tid % tpr;
  float o[G][8];
#pragma unroll
  for (int g = 0; g < G; ++g)
#pragma unroll
    for (int e = 0; e < 8; ++e) o[g][e] = 0.f;
  if (r < rows) {
    for (int pb = p0 + r; pb < p1; pb += 4 * rows) {  // four rows of V in flight per thread
      uint4 vv[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int p = pb + j * rows;
        vv[j] = p < p1 ? *reinterpret_cast<const uint4*>(vc + (size_t)(p % L) * D + dc * 8) : make_uint4(0u, 0u, 0u, 0u);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int p = pb + j * rows;
        if (p >= p1) break;
        float vf[8];
        unpack8<T>(vv[j], vf);
#pragma unroll
        for (int g = 0; g < G; ++g) {
          const float pr = sc[g * a.chunk + (p - p0)];
#pragma unroll
          for (int e = 0; e < 8; ++e) o[g][e] = fmaf(pr, vf[e], o[g][e]);
        }
      }
    }
  }
  // reduce over the position rows through shared memory (reusing the logits' space: every probability has been read)
  __syncthreads();
  float* pv = sc;  // [rows][G][D]
  if (r < rows) {
#pragma unroll
    for (int g = 0; g < G; ++g)
#pragma unroll
      for (int e = 0; e < 8; ++e) pv[(r * G + g) * D + dc * 8 + e] = o[g][e];
  }
  __syncthreads();
  att_finish<T>(a, G, b, kvh, split, stat, stat + G, [&](int i) {
    float s = 0.f;
    for (int rr = 0; rr < rows; ++rr) s += pv[rr * G * D + i];
    return s;
  });
}

// ------------------------------------------------------------------------------------------ wide groups: tensor cores
// mma.sync m16n8k16 (row.col, fp32 accumulate).  Warp (mt, pg) owns head rows mt * 16 .. + 15 of the G_pad = 16 * MT
// rows and every PG-th block of 16 positions of the chunk; it keeps an online softmax (max, sum) per row and the
// unnormalised output rows in registers.  The PG partial results of a row are merged through shared memory at the end.
//
// Channel orders.  Q.K^T: lane (r8 = lane / 4, q4 = lane % 4) of a 16-position block loads ONE uint4 of K per n-tile
// and per 32 channels: position pb + 8 t + r8, channels 32 ch + 8 q4 .. + 7.  Its four words are b0 / b1 of the k-steps
// (ch, s = 0) and (ch, s = 1), so the k index of step (ch, s) maps to channel
//   kidx = 32 ch + 16 s + 8 hi + 2 q4 + j   <->   channel 32 ch + 8 q4 + 4 s + 2 hi + j        (att_tc_kidx)
// and Q is stored in shared memory by kidx, so that a plain ldmatrix.x4 yields the matching A fragment.
// P.V: the C fragment of Q.K^T is the A fragment of P.V (k index kk <-> position pb + kk).  Lane (r8, q4) loads rows
// pb + 2 q4, + 1, + 8, + 9 of V at channels 64 v + 8 r8 .. + 7 and pairs them up with byte permutes: n-tile e of the
// 64-channel slab v then holds channel 64 v + 8 n + e in column n, and the output fragment of that n-tile covers
// channels 64 v + 16 q4 + e (c0, c2) and 64 v + 16 q4 + 8 + e (c1, c3).
// K and V are read with ordinary (generic-proxy, coherent) loads: the __syncthreads() after the current-step prologue
// orders this CTA's own cache-slot writes before them.
constexpr int kTcWarps = kAttThreads / 32;

__device__ __forceinline__ int att_tc_kidx(int c) {
  return (c & ~31) + ((c >> 2) & 1) * 16 + ((c >> 1) & 1) * 8 + ((c >> 3) & 3) * 2 + (c & 1);
}

template <typename T>
__device__ __forceinline__ uint32_t pack2_rn(float lo, float hi) {
  if constexpr (TypeTraits<T>::kIsBf16) return b2_as_u32(__floats2bfloat162_rn(lo, hi));
  else return h2_as_u32(__floats2half2_rn(lo, hi));
}

__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
               : "r"(addr));
}

__device__ __forceinline__ uint32_t u4_word(const uint4& v, int i) { return i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w; }

// shared memory of the tensor-core kernel, in floats: [max(query tile, PG partial outputs)] [PG][GP] max [PG][GP] sum
// [GP] chunk max [GP] chunk sum
struct AttTcSmem {
  int MT, GP, PG, qstride, region;
  __host__ __device__ AttTcSmem(int G, int D) {
    MT = (G + 15) / 16, GP = MT * 16, PG = kTcWarps / MT;
    qstride = (D + 31) / 32 * 32 + 8;  // T elements per query row: 16 bytes of padding keep ldmatrix conflict-free
    const int qfloats = GP * qstride / 2, ofloats = PG * GP * D;
    region = qfloats > ofloats ? qfloats : ofloats;
  }
  __host__ __device__ size_t bytes() const { return ((size_t)region + 2 * PG * GP + 2 * GP) * sizeof(float); }
};

// NV = ceil(D / 64): 64-channel slabs of V (and of the output) per lane
template <typename T, int NV>
__global__ void __launch_bounds__(kAttThreads) single_query_attention_tc_kernel(const AttArgs a) {
  extern __shared__ __align__(16) float att_smem[];
  const int D = a.D, L = a.L, G = a.H / a.Hkv;
  const AttTcSmem lay(G, D);
  const int GP = lay.GP, PG = lay.PG, QS = lay.qstride;
  T* qs = reinterpret_cast<T*>(att_smem);  // [GP][QS] rotated, rounded queries in kidx order; zero where g >= G or c >= D
  float* co = att_smem;                    // after the loop: [PG][GP][D] partial outputs (over the queries)
  float* cm = att_smem + lay.region;       // [PG][GP] running max -> merge weight
  float* cl = cm + PG * GP;                // [PG][GP] sum
  float* stat = cl + PG * GP;              // [GP] max, [GP] sum of the chunk
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, r8 = lane >> 2, q4 = lane & 3;
  const int split = blockIdx.x, kvh = blockIdx.y, b = blockIdx.z;
  const T* kc = static_cast<const T*>(a.k_cache) + (size_t)(b * a.Hkv + kvh) * L * D;
  const T* vc = static_cast<const T*>(a.v_cache) + (size_t)(b * a.Hkv + kvh) * L * D;
  for (int i = tid; i < GP * QS / 2; i += kAttThreads) reinterpret_cast<uint32_t*>(qs)[i] = 0u;
  pdl_launch_dependents();
  pdl_wait_prior_grid();
  const int tlength = a.length_per_sample ? a.length_per_sample[b] : a.timestep;
  const int first = max(0, tlength + 1 - L);
  const int npos = tlength + 1 - first;
  const int p0 = first + split * a.chunk, p1 = min(first + npos, p0 + a.chunk);
  const bool has_current = p0 <= tlength && tlength < p0 + a.chunk;
  __syncthreads();  // the zero fill lands before the queries
  att_current_step<T>(a, G, b, kvh, tlength, has_current, [&](int g, int c, T x) { qs[g * QS + att_tc_kidx(c)] = x; });
  __syncthreads();  // qs complete; this CTA's own cache writes are visible to its own reads below

  const int mt = warp % lay.MT, pg = warp / lay.MT;
  const int ncg = D >> 3;  // 8-channel groups
  float o[NV][8][4];
#pragma unroll
  for (int v = 0; v < NV; ++v)
#pragma unroll
    for (int e = 0; e < 8; ++e) o[v][e][0] = o[v][e][1] = o[v][e][2] = o[v][e][3] = 0.f;
  float m0 = -FLT_MAX, m1 = -FLT_MAX, l0 = 0.f, l1 = 0.f;  // rows r8 and r8 + 8 of this warp's tile
  if (pg < PG) {
    // ldmatrix.x4 addresses: lanes 0-7 rows 0-7 / 8-15 rows 8-15 at k 0-7, lanes 16-31 the same rows at k 8-15
    const uint32_t qaddr = smem_u32(qs) + ((mt * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * QS + (lane >> 4) * 8) * 2;
    const int nblk = (p1 - p0 + 15) >> 4;
    for (int blk = pg; blk < nblk; blk += PG) {
      const int pb = p0 + blk * 16;
      // ---- logits S[16 rows][16 positions]: s[t] is n-tile t (positions pb + 8 t ..); K is loaded 32 channels at a time
      const T* kp0 = kc + (size_t)((pb + r8) % L) * 8;
      const T* kp1 = kc + (size_t)((pb + 8 + r8) % L) * 8;
      const bool kin0 = pb + r8 < p1, kin1 = pb + 8 + r8 < p1;
      float s[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
      for (int ch = 0; ch < 2 * NV; ++ch) {
        if (32 * ch >= D) break;
        const int grp = 4 * ch + q4;
        const uint4 z = make_uint4(0u, 0u, 0u, 0u);
        const uint4 k0 = kin0 && grp < ncg ? *reinterpret_cast<const uint4*>(kp0 + (size_t)grp * L * 8) : z;
        const uint4 k1 = kin1 && grp < ncg ? *reinterpret_cast<const uint4*>(kp1 + (size_t)grp * L * 8) : z;
#pragma unroll
        for (int st = 0; st < 2; ++st) {
          uint32_t a0, a1, a2, a3;
          ldsm_x4(qaddr + (ch * 32 + st * 16) * 2, a0, a1, a2, a3);
          mma_16816<T>(s[0], a0, a1, a2, a3, u4_word(k0, 2 * st), u4_word(k0, 2 * st + 1), s[0]);
          mma_16816<T>(s[1], a0, a1, a2, a3, u4_word(k1, 2 * st), u4_word(k1, 2 * st + 1), s[1]);
        }
      }
      // ---- online softmax: c0 / c1 of an n-tile are row r8, c2 / c3 row r8 + 8, positions pb + 8 t + 2 q4 + (0, 1)
      float bm0 = -INFINITY, bm1 = -INFINITY;
#pragma unroll
      for (int t = 0; t < 2; ++t)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int p = pb + 8 * t + 2 * q4 + (j & 1);
          s[t][j] = p < p1 ? s[t][j] * a.inv_sqrt_d : -INFINITY;
          if (j < 2) bm0 = fmaxf(bm0, s[t][j]);
          else bm1 = fmaxf(bm1, s[t][j]);
        }
#pragma unroll
      for (int x = 1; x < 4; x <<= 1) {
        bm0 = fmaxf(bm0, __shfl_xor_sync(0xffffffffu, bm0, x));
        bm1 = fmaxf(bm1, __shfl_xor_sync(0xffffffffu, bm1, x));
      }
      const float n0 = fmaxf(m0, bm0), n1 = fmaxf(m1, bm1);
      const float c0 = __expf(m0 - n0), c1 = __expf(m1 - n1);
      m0 = n0, m1 = n1;
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        s[t][0] = __expf(s[t][0] - n0), s[t][1] = __expf(s[t][1] - n0);
        s[t][2] = __expf(s[t][2] - n1), s[t][3] = __expf(s[t][3] - n1);
      }
      l0 = fmaf(l0, c0, (s[0][0] + s[0][1]) + (s[1][0] + s[1][1]));
      l1 = fmaf(l1, c1, (s[0][2] + s[0][3]) + (s[1][2] + s[1][3]));
      // ---- P (rounded to T) x V
      const uint32_t pa0 = pack2_rn<T>(s[0][0], s[0][1]), pa1 = pack2_rn<T>(s[0][2], s[0][3]);
      const uint32_t pa2 = pack2_rn<T>(s[1][0], s[1][1]), pa3 = pack2_rn<T>(s[1][2], s[1][3]);
#pragma unroll
      for (int v = 0; v < NV; ++v) {  // V one 64-channel slab at a time
        if (64 * v >= D) break;
        uint4 vr[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int p = pb + 2 * q4 + (j & 1) + 8 * (j >> 1);
          vr[j] = p < p1 && 8 * v + r8 < ncg ? *reinterpret_cast<const uint4*>(vc + (size_t)(p % L) * D + v * 64 + r8 * 8)
                                             : make_uint4(0u, 0u, 0u, 0u);
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const unsigned sel = (e & 1) ? 0x7632u : 0x5410u;
          const uint32_t b0 = __byte_perm(u4_word(vr[0], e >> 1), u4_word(vr[1], e >> 1), sel);
          const uint32_t b1 = __byte_perm(u4_word(vr[2], e >> 1), u4_word(vr[3], e >> 1), sel);
          o[v][e][0] *= c0, o[v][e][1] *= c0, o[v][e][2] *= c1, o[v][e][3] *= c1;
          mma_16816<T>(o[v][e], pa0, pa1, pa2, pa3, b0, b1, o[v][e]);
        }
      }
    }
  }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1), l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1), l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  __syncthreads();  // every warp is done with qs: the partial outputs overlay it
  if (pg < PG) {
    const int row = mt * 16 + r8;
    float* o0 = co + ((size_t)pg * GP + row) * D;
    float* o1 = o0 + 8 * D;
#pragma unroll
    for (int v = 0; v < NV; ++v)
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int d = 64 * v + 16 * q4 + e;
        if (d < D) o0[d] = o[v][e][0], o1[d] = o[v][e][2];
        if (d + 8 < D) o0[d + 8] = o[v][e][1], o1[d + 8] = o[v][e][3];
      }
    if (q4 == 0) {
      cm[pg * GP + row] = m0, cm[pg * GP + row + 8] = m1;
      cl[pg * GP + row] = l0, cl[pg * GP + row + 8] = l1;
    }
  }
  __syncthreads();
  // merge the PG partials of each real head row (rows G .. GP - 1 are padding: never read)
  for (int g = tid; g < G; g += kAttThreads) {
    float M = -FLT_MAX;
    for (int w = 0; w < PG; ++w) M = fmaxf(M, cm[w * GP + g]);
    float sum = 0.f;
    for (int w = 0; w < PG; ++w) {
      const float wt = __expf(cm[w * GP + g] - M);
      cm[w * GP + g] = wt;
      sum = fmaf(wt, cl[w * GP + g], sum);
    }
    stat[g] = M, stat[GP + g] = sum;
  }
  __syncthreads();
  att_finish<T>(a, G, b, kvh, split, stat, stat + GP, [&](int i) {
    const int g = i / D, d = i - g * D;
    float s = 0.f;
    for (int w = 0; w < PG; ++w) s = fmaf(cm[w * GP + g], co[((size_t)w * GP + g) * D + d], s);
    return s;
  });
}

template <typename T>
const void* att_kernel_small(int G) {
  switch (G) {
    case 1: return (const void*)single_query_attention_kernel<T, 1>;
    case 2: return (const void*)single_query_attention_kernel<T, 2>;
    case 3: return (const void*)single_query_attention_kernel<T, 3>;
    case 4: return (const void*)single_query_attention_kernel<T, 4>;
    case 5: return (const void*)single_query_attention_kernel<T, 5>;
    case 6: return (const void*)single_query_attention_kernel<T, 6>;
    case 7: return (const void*)single_query_attention_kernel<T, 7>;
    case 8: return (const void*)single_query_attention_kernel<T, 8>;
    default: return nullptr;
  }
}

template <typename T>
const void* att_kernel_tc(int D) {
  switch ((D + 63) / 64) {
    case 1: return (const void*)single_query_attention_tc_kernel<T, 1>;
    case 2: return (const void*)single_query_attention_tc_kernel<T, 2>;
    case 3: return (const void*)single_query_attention_tc_kernel<T, 3>;
    case 4: return (const void*)single_query_attention_tc_kernel<T, 4>;
    default: return nullptr;
  }
}

int launch_att(const void* kern, const AttArgs& a, size_t smem, bool pdl, cudaStream_t stream) {
  if (!kern) return B200AWQ_ERR_SHAPE;
  if (smem > 48 * 1024) {
    if (cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) return (int)e;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)a.splits, (unsigned)a.Hkv, (unsigned)a.B);
  cfg.blockDim = dim3(kAttThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  void* args[] = {const_cast<AttArgs*>(&a)};
  cudaError_t e = cudaLaunchKernelExC(&cfg, kern, args);
  return e == cudaSuccess ? 0 : (int)e;
}

// ------------------------------------------------------------------------------------------------ RoPE over [s, b, h, d]
struct RopeArgs {
  const void* x;
  const float* freqs;
  void* y;
  int s, b, h, d, d2;
  long long ss, sb, sh, sd, os, ob, oh, od;
};

template <typename T>
__global__ void __launch_bounds__(256) rope_with_pos_kernel(const RopeArgs a) {
  pdl_launch_dependents();
  pdl_wait_prior_grid();
  const int s_id = blockIdx.x, b_id = blockIdx.y;
  const T* src = static_cast<const T*>(a.x) + s_id * a.ss + b_id * a.sb;
  T* dst = static_cast<T*>(a.y) + s_id * a.os + b_id * a.ob;
  const float* fr = a.freqs + ((size_t)b_id * a.s + s_id) * a.d2;  // fused_rope_with_pos.cu:46
  for (int i = threadIdx.x; i < a.h * a.d; i += blockDim.x) {
    const int h_id = i / a.d, d_id = i % a.d;
    const T* sp = src + h_id * a.sh;
    float v = t2f<T>(sp[d_id * a.sd]);
    if (d_id < a.d2) {
      float sn, cs;
      sincosf(fr[d_id], &sn, &cs);
      const float rot = (d_id + a.d2 / 2 < a.d2) ? -t2f<T>(sp[(d_id + a.d2 / 2) * a.sd]) : t2f<T>(sp[(d_id - a.d2 / 2) * a.sd]);
      v = v * cs + rot * sn;  // fused_rope_with_pos.cu:52-57
    }
    dst[h_id * a.oh + d_id * a.od] = from_float<T>(v);
  }
}

}  // namespace

size_t attention_workspace_bytes(int batch, int heads, int kv_heads, int head_dim, int max_len) {
  if (batch < 1 || kv_heads < 1 || heads < kv_heads || head_dim < 8) return 0;
  const int G = heads / kv_heads;
  const size_t max_splits = 64;
  (void)max_len;
  // [counters: kAttCounters x u32, always at offset 0 whatever the shape -- partials of an earlier launch with another
  // shape must never alias them] [partials]
  return kAttCounters * sizeof(unsigned int) + (size_t)batch * kv_heads * (max_splits * G * (head_dim + 2) * sizeof(float));
}

int launch_single_query_attention(const void* q, const void* k, const void* v, void* k_cache, void* v_cache, void* out,
                                  const int* length_per_sample, int batch, int heads, int kv_heads, int head_dim, int max_len,
                                  int timestep, long long q_batch_stride, long long k_batch_stride, long long v_batch_stride, int rotary_dim, float rotary_base, float rotary_scale,
                                  int neox, int dtype, void* workspace, size_t workspace_bytes, bool pdl, cudaStream_t stream) {
  if (batch < 1 || kv_heads < 1 || heads % kv_heads || head_dim % 8 || head_dim > kAttMaxD || max_len < 1 || timestep < 0 ||
      rotary_dim < 0 || rotary_dim > head_dim || (rotary_dim & 1) || (neox && rotary_dim % 2))
    return B200AWQ_ERR_SHAPE;
  const int G = heads / kv_heads;
  const bool tc = G > kAttMaxG;  // wide groups: tensor cores
  if (G > kAttTcMaxG || (tc && head_dim % 16) || (long long)batch * kv_heads > kAttCounters) return B200AWQ_ERR_SHAPE;
  if (workspace_bytes < attention_workspace_bytes(batch, heads, kv_heads, head_dim, max_len) || !workspace)
    return B200AWQ_ERR_WORKSPACE;
  AttArgs a{};
  a.q = q, a.k = k, a.v = v, a.k_cache = k_cache, a.v_cache = v_cache, a.out = out;
  a.length_per_sample = length_per_sample;
  a.B = batch, a.H = heads, a.Hkv = kv_heads, a.D = head_dim, a.L = max_len, a.timestep = timestep;
  a.q_stride = q_batch_stride, a.k_stride = k_batch_stride, a.v_stride = v_batch_stride;
  a.rot_dim = rotary_dim, a.neox = neox, a.base = rotary_base, a.scale = rotary_scale;
  a.inv_sqrt_d = 1.f / sqrtf((float)head_dim);
  // worst-case positions (length_per_sample is on the device): the chunking must cover up to min(timestep, max_len - 1) + 1
  const int npos_max = std::min(length_per_sample ? max_len : timestep + 1, max_len);
  int dev = 0, nsm = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
  int splits = std::max(1, std::min(64, 2 * nsm / std::max(1, batch * kv_heads)));
  splits = std::min(splits, (npos_max + 127) / 128);                  // >= 128 positions per CTA
  if (!tc) {                                                          // the logits of a chunk live in shared memory
    const int chunk_cap = std::max(256, (48 * 1024 / 4) / G / 32 * 32);  // G * chunk floats <= 48 KB
    splits = std::max(splits, (npos_max + chunk_cap - 1) / chunk_cap);
  }
  if (splits > 64) return B200AWQ_ERR_SHAPE;
  a.splits = std::max(1, splits);
  a.chunk = ((npos_max + a.splits - 1) / a.splits + 31) / 32 * 32;
  a.count = static_cast<unsigned int*>(workspace);
  a.ws = reinterpret_cast<float*>(static_cast<char*>(workspace) + kAttCounters * sizeof(unsigned int));
  const bool f16 = dtype == B200AWQ_DTYPE_F16;
  if (tc) {
    const size_t smem = AttTcSmem(G, head_dim).bytes();
    if (smem > 200 * 1024) return B200AWQ_ERR_SHAPE;
    return launch_att(f16 ? att_kernel_tc<__half>(head_dim) : att_kernel_tc<__nv_bfloat16>(head_dim), a, smem, pdl, stream);
  }
  // position rows of the P.V loop: D / 8 threads per row, the remainder of the 256 threads idle
  const int rows = kAttThreads / (head_dim / 8);
  const size_t sc_floats = std::max((size_t)G * a.chunk, (size_t)rows * G * head_dim);
  const size_t smem = ((size_t)G * head_dim + kAttThreads / 32 * G + 2 * G + sc_floats) * sizeof(float) + 16;
  if (smem > 200 * 1024) return B200AWQ_ERR_SHAPE;
  return launch_att(f16 ? att_kernel_small<__half>(G) : att_kernel_small<__nv_bfloat16>(G), a, smem, pdl, stream);
}

int launch_rope_with_pos(const void* x, const float* freqs, void* y, int s, int b, int h, int d, int d2, const long long* in_strides,
                         const long long* out_strides, int dtype, bool pdl, cudaStream_t stream) {
  if (s < 1 || b < 1 || h < 1 || d < 1 || d2 < 0 || d2 > d || (d2 & 1)) return B200AWQ_ERR_SHAPE;
  RopeArgs a{x, freqs, y, s, b, h, d, d2, in_strides[0], in_strides[1], in_strides[2], in_strides[3],
             out_strides[0], out_strides[1], out_strides[2], out_strides[3]};
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)s, (unsigned)b);
  cfg.blockDim = dim3(256);
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  cudaError_t e;
  if (dtype == B200AWQ_DTYPE_F16) e = cudaLaunchKernelEx(&cfg, rope_with_pos_kernel<__half>, a);
  else e = cudaLaunchKernelEx(&cfg, rope_with_pos_kernel<__nv_bfloat16>, a);
  return e == cudaSuccess ? 0 : (int)e;
}

}  // namespace b200awq
