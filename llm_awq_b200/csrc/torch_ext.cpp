// Python module `awq_inference_engine`: the reference's extension name and the two entry
// points WQLinear / tinychat call (awq/kernels/csrc/pybind.cpp:22-23), as a thin shim over
// the C ABI in include/b200awq.h.  Same positional signatures, same return tensors, same
// exception types as the reference host functions (gemv_cuda.cu:245-338,
// gemm_cuda.cu:1126-1236); additionally: launches on the CURRENT stream of the input's
// device (the reference uses the legacy default stream and no device guard), checks
// contiguity / shapes, and surfaces launch errors.
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/extension.h>

#include <map>
#include <stdexcept>

#include "../../include/b200awq.h"

namespace {

int dtype_code(const torch::Tensor& t, const char* fn) {
  if (t.scalar_type() == at::ScalarType::Half) return B200AWQ_DTYPE_F16;
  if (t.scalar_type() == at::ScalarType::BFloat16) return B200AWQ_DTYPE_BF16;
  // reference: dispatch_utils.cuh:13-17
  TORCH_CHECK(false, fn, " failed to dispatch data type ", t.scalar_type());
}

void check_inputs(const torch::Tensor& in, const torch::Tensor& kernel, const torch::Tensor& scales,
                  const torch::Tensor& zeros) {
  TORCH_CHECK(in.is_cuda() && kernel.is_cuda() && scales.is_cuda() && zeros.is_cuda(), "all tensors must be CUDA tensors");
  TORCH_CHECK(scales.scalar_type() == in.scalar_type());  // reference: gemv_cuda.cu:260, gemm_cuda.cu:1145
  TORCH_CHECK(zeros.scalar_type() == in.scalar_type());   // reference: gemv_cuda.cu:261, gemm_cuda.cu:1146
  TORCH_CHECK(kernel.scalar_type() == at::ScalarType::Short, "qweight must be int16 [N/4, K]");
  TORCH_CHECK(in.is_contiguous() && kernel.is_contiguous() && scales.is_contiguous() && zeros.is_contiguous(),
              "inputs must be contiguous");
  TORCH_CHECK(kernel.dim() == 2 && scales.dim() == 2 && zeros.dim() == 2 && in.dim() >= 1, "bad tensor ranks");
}

void raise(int code, bool is_gemv) {
  if (code == 0) return;
  // the reference throws std::runtime_error for unsupported batch / group (gemv_cuda.cu:329,334)
  if (is_gemv && code == B200AWQ_ERR_BATCH) throw std::runtime_error("Unsupported batch size for gemv kernel.\n");
  if (is_gemv && code == B200AWQ_ERR_GROUP) throw std::runtime_error("Unsupported group size for gemv kernel.\n");
  TORCH_CHECK(false, "b200awq: ", b200awq_strerror(code), " (code ", code, ")");
}

}  // namespace

torch::Tensor gemv_forward_cuda_new(torch::Tensor _in_feats, torch::Tensor _kernel, torch::Tensor _scaling_factors,
                                    torch::Tensor _zeros, int m, int n, int k, int group_size) {
  check_inputs(_in_feats, _kernel, _scaling_factors, _zeros);
  const int dt = dtype_code(_in_feats, "gemv_forward_cuda_new");
  TORCH_CHECK(_in_feats.size(-1) == k && _in_feats.numel() == (int64_t)m * k, "in_feats does not match (m, k)");
  TORCH_CHECK(_kernel.size(0) * 4 == n && _kernel.size(1) == k, "qweight does not match (n, k)");
  TORCH_CHECK(_scaling_factors.size(1) == n && _zeros.size(1) == n && _scaling_factors.size(0) * group_size >= k &&
                  _zeros.size(0) * group_size >= k,
              "scales / zeros do not match (n, k, group)");
  const c10::cuda::CUDAGuard guard(_in_feats.device());
  std::vector<int64_t> output_shape = _in_feats.sizes().vec();
  output_shape.back() = n;
  at::Tensor out = torch::empty(output_shape, _in_feats.options());
  raise(b200awq_w4a16_gemv(_in_feats.data_ptr(), _kernel.data_ptr(), _scaling_factors.data_ptr(), _zeros.data_ptr(),
                           out.data_ptr(), m, n, k, group_size, dt, at::cuda::getCurrentCUDAStream().stream()),
        true);
  return out;
}

torch::Tensor gemm_forward_cuda_new(torch::Tensor _in_feats, torch::Tensor _kernel, torch::Tensor _scales,
                                    torch::Tensor _zeros) {
  check_inputs(_in_feats, _kernel, _scales, _zeros);
  const int dt = dtype_code(_in_feats, "gemm_forward_cuda_new");
  const int64_t k = _in_feats.size(-1);
  const int64_t n = _kernel.size(0) * 4;  // reference: gemm_cuda.cu:1133
  const int64_t m = _in_feats.numel() / k;
  TORCH_CHECK(_kernel.size(1) == k, "qweight does not match in_feats");
  TORCH_CHECK(_scales.size(1) == n && _zeros.size(1) == n && _scales.size(0) * 128 >= k && _zeros.size(0) * 128 >= k,
              "scales / zeros do not match (n, k)");
  const c10::cuda::CUDAGuard guard(_in_feats.device());
  std::vector<int64_t> output_shape = _in_feats.sizes().vec();
  output_shape.back() = n;
  at::Tensor out = torch::empty(output_shape, _in_feats.options());
  if (m == 0) return out;
  const size_t ws_bytes = b200awq_w4a16_gemm_workspace_bytes((int)m, (int)n, (int)k);
  at::Tensor ws;
  if (ws_bytes) ws = torch::empty({(int64_t)ws_bytes}, _in_feats.options().dtype(torch::kUInt8));
  raise(b200awq_w4a16_gemm(_in_feats.data_ptr(), _kernel.data_ptr(), _scales.data_ptr(), _zeros.data_ptr(), out.data_ptr(),
                           (int)m, (int)n, (int)k, 128, dt, ws_bytes ? ws.data_ptr() : nullptr, ws_bytes,
                           at::cuda::getCurrentCUDAStream().stream()),
        false);
  return out;
}

// New entry (no counterpart in the reference's extension): the whole of QuantLlamaMLP.our_llama_mlp
// (tinychat/modules/fused_mlp.py:36-83) in one call.  The zeros tensors are used as given.
torch::Tensor mlp_front_forward_cuda(torch::Tensor _in_feats, torch::Tensor _gate_kernel, torch::Tensor _gate_scales,
                                     torch::Tensor _gate_zeros, torch::Tensor _up_kernel, torch::Tensor _up_scales,
                                     torch::Tensor _up_zeros) {
  check_inputs(_in_feats, _gate_kernel, _gate_scales, _gate_zeros);
  check_inputs(_in_feats, _up_kernel, _up_scales, _up_zeros);
  const int dt = dtype_code(_in_feats, "mlp_front_forward_cuda");
  const int64_t k = _in_feats.size(-1);
  const int64_t n = _gate_kernel.size(0) * 4;
  const int64_t m = _in_feats.numel() / k;
  TORCH_CHECK(_gate_kernel.size(1) == k && _up_kernel.size(0) * 4 == n && _up_kernel.size(1) == k, "qweights do not match");
  for (const torch::Tensor* t : {&_gate_scales, &_gate_zeros, &_up_scales, &_up_zeros})
    TORCH_CHECK(t->size(1) == n && t->size(0) * 128 >= k, "scales / zeros do not match (n, k)");
  const c10::cuda::CUDAGuard guard(_in_feats.device());
  std::vector<int64_t> output_shape = _in_feats.sizes().vec();
  output_shape.back() = n;
  at::Tensor out = torch::empty(output_shape, _in_feats.options());
  if (m == 0) return out;
  at::Tensor ws;
  size_t ws_bytes = 0;
  if (!(m == 1 && dt == B200AWQ_DTYPE_F16)) {
    ws_bytes = b200awq_w4a16_mlp_front_workspace_bytes((int)m, (int)n, (int)k);
    ws = torch::empty({(int64_t)ws_bytes}, _in_feats.options().dtype(torch::kUInt8));
  }
  int rc = b200awq_w4a16_mlp_front(_in_feats.data_ptr(), _gate_kernel.data_ptr(), _gate_scales.data_ptr(), _gate_zeros.data_ptr(),
                                   _up_kernel.data_ptr(), _up_scales.data_ptr(), _up_zeros.data_ptr(), out.data_ptr(), (int)m,
                                   (int)n, (int)k, 128, dt, ws_bytes ? ws.data_ptr() : nullptr, ws_bytes,
                                   at::cuda::getCurrentCUDAStream().stream());
  if (rc == B200AWQ_ERR_WORKSPACE && ws_bytes == 0) {  // the one-kernel path declined the shape: composed path
    ws_bytes = b200awq_w4a16_mlp_front_workspace_bytes((int)m, (int)n, (int)k);
    ws = torch::empty({(int64_t)ws_bytes}, _in_feats.options().dtype(torch::kUInt8));
    rc = b200awq_w4a16_mlp_front(_in_feats.data_ptr(), _gate_kernel.data_ptr(), _gate_scales.data_ptr(), _gate_zeros.data_ptr(),
                                 _up_kernel.data_ptr(), _up_scales.data_ptr(), _up_zeros.data_ptr(), out.data_ptr(), (int)m, (int)n,
                                 (int)k, 128, dt, ws.data_ptr(), ws_bytes, at::cuda::getCurrentCUDAStream().stream());
  }
  raise(rc, false);
  return out;
}

// reference: awq/kernels/csrc/layernorm/layernorm.cu:111-131 (input [b, s, c], gamma [c], out like input; returns
// nothing).  Same dtype checks; additionally any rank >= 1 is accepted (rows = numel / last dim), the launch goes to
// the current stream, and contiguity is checked instead of assumed.
void layernorm_forward_cuda(torch::Tensor _input, torch::Tensor _gamma, torch::Tensor _out, float eps) {
  TORCH_CHECK(_input.is_cuda() && _gamma.is_cuda() && _out.is_cuda(), "all tensors must be CUDA tensors");
  const int dt = dtype_code(_input, "layernorm_forward_cuda");
  TORCH_CHECK(_gamma.scalar_type() == _input.scalar_type());  // layernorm.cu:122
  TORCH_CHECK(_out.scalar_type() == _input.scalar_type());    // layernorm.cu:123
  TORCH_CHECK(_input.dim() >= 1 && _input.is_contiguous() && _out.is_contiguous() && _gamma.is_contiguous(),
              "inputs must be contiguous");
  const int64_t n = _input.size(-1);
  TORCH_CHECK(_gamma.numel() == n && _out.numel() == _input.numel(), "gamma / out do not match input");
  if (_input.numel() == 0) return;
  const c10::cuda::CUDAGuard guard(_input.device());
  raise(b200awq_rmsnorm(_input.data_ptr(), _gamma.data_ptr(), _out.data_ptr(), (int)(_input.numel() / n), (int)n, eps, dt,
                        at::cuda::getCurrentCUDAStream().stream()),
        false);
}

// reference: awq/kernels/csrc/attention/ft_attention.cpp:112-184 (same checks, same argument order and defaults,
// pybind.cpp:24-27).  Any nheads / nheads_kv ratio up to 128 (the GQA / multi-query callers of Qwen2, Llama-3.2,
// Falcon); the head_dim limits are those of b200awq_single_query_attention.  alibi_slopes must be None; fp32 tensors are
// not dispatched.
torch::Tensor single_query_attention(const torch::Tensor q, const torch::Tensor k, const torch::Tensor v, torch::Tensor k_cache,
                                     torch::Tensor v_cache, c10::optional<const torch::Tensor> length_per_sample_,
                                     c10::optional<const torch::Tensor> alibi_slopes_, const int timestep,
                                     const int rotary_embedding_dim, const float rotary_base, const float rotary_scale,
                                     const bool neox_rotary_style) {
  TORCH_CHECK(q.is_cuda() && k.is_cuda() && v.is_cuda() && k_cache.is_cuda() && v_cache.is_cuda(), "tensors must be on CUDA");
  const int batch_size = v_cache.size(0), nheads = q.size(1), nheads_kv = v_cache.size(1);
  const int memory_max_seqlen = v_cache.size(2), headdim = v_cache.size(3);
  TORCH_CHECK(q.sizes() == torch::IntArrayRef({batch_size, nheads, headdim}), "q must have shape (batch, nheads, headdim)");
  TORCH_CHECK(k.sizes() == torch::IntArrayRef({batch_size, nheads_kv, headdim}), "k must have shape (batch, nheads_kv, headdim)");
  TORCH_CHECK(v.sizes() == torch::IntArrayRef({batch_size, nheads_kv, headdim}), "v must have shape (batch, nheads_kv, headdim)");
  TORCH_CHECK(k_cache.sizes() == torch::IntArrayRef({batch_size, nheads_kv, headdim / 8, memory_max_seqlen, 8}),
              "k_cache must have shape (batch, nheads_kv, headdim / 8, max_seqlen, 8)");
  TORCH_CHECK(q.stride(2) == 1 && q.stride(1) == headdim);
  TORCH_CHECK(k.stride(2) == 1 && k.stride(1) == headdim);
  TORCH_CHECK(v.stride(2) == 1 && v.stride(1) == headdim);
  TORCH_CHECK(v_cache.is_contiguous() && k_cache.is_contiguous(), "caches must be contiguous");
  const int dt = dtype_code(q, "single_query_attention");
  TORCH_CHECK(k.scalar_type() == q.scalar_type() && v.scalar_type() == q.scalar_type() &&
              k_cache.scalar_type() == q.scalar_type() && v_cache.scalar_type() == q.scalar_type());
  TORCH_CHECK(!alibi_slopes_.has_value(), "b200awq: alibi_slopes is not supported by this build");
  const int* lps = nullptr;
  if (length_per_sample_.has_value()) {
    const auto& l = length_per_sample_.value();
    TORCH_CHECK(l.is_cuda() && l.is_contiguous() && l.dtype() == torch::kInt32 && l.numel() == batch_size);
    lps = l.data_ptr<int>();
  }
  const c10::cuda::CUDAGuard guard(q.device());
  torch::Tensor out = torch::empty({batch_size, nheads, headdim}, q.options());
  // one zero-initialised workspace per (device, stream); the kernels leave it zero where it matters
  // (leaked on purpose: CUDA tensors must not be destroyed by static destructors at interpreter exit)
  static auto& workspaces = *new std::map<std::pair<int, void*>, torch::Tensor>();
  const size_t need = b200awq_single_query_attention_workspace_bytes(batch_size, nheads, nheads_kv, headdim, memory_max_seqlen);
  void* st = at::cuda::getCurrentCUDAStream().stream();
  auto key = std::make_pair((int)q.get_device(), st);
  auto it = workspaces.find(key);
  if (it == workspaces.end() || (size_t)it->second.numel() < need) {
    workspaces[key] = torch::zeros({(int64_t)need}, q.options().dtype(torch::kUInt8));
    it = workspaces.find(key);
  }
  raise(b200awq_single_query_attention(q.data_ptr(), k.data_ptr(), v.data_ptr(), k_cache.data_ptr(), v_cache.data_ptr(),
                                       out.data_ptr(), lps, batch_size, nheads, nheads_kv, headdim, memory_max_seqlen, timestep,
                                       (long long)q.stride(0), (long long)k.stride(0), (long long)v.stride(0), rotary_embedding_dim, rotary_base, rotary_scale,
                                       neox_rotary_style ? 1 : 0, dt, it->second.data_ptr(), (size_t)it->second.numel(), st),
        false);
  return out;
}

// reference: awq/kernels/csrc/rope_new/fused_rope_with_pos.cu:243-285
at::Tensor fused_rope_with_pos_forward_func(const at::Tensor& input, const at::Tensor& freqs, const bool transpose_output_memory) {
  TORCH_CHECK(input.is_cuda() && freqs.is_cuda() && input.dim() == 4, "input must be a CUDA tensor [s, b, h, d]");
  TORCH_CHECK(freqs.scalar_type() == at::ScalarType::Float && freqs.is_contiguous(), "freqs must be contiguous float32");
  const int dt = dtype_code(input, "fused_rope_with_pos_forward_func");
  const int s = input.size(0), b = input.size(1), h = input.size(2), d = input.size(3), d2 = freqs.size(-1);
  TORCH_CHECK(freqs.numel() >= (int64_t)s * b * d2, "freqs must hold s * b * d2 angles");
  auto opts = input.options().requires_grad(false);
  at::Tensor output = transpose_output_memory ? torch::empty({b, s, h, d}, opts).transpose(0, 1) : torch::empty({s, b, h, d}, opts);
  const long long is[4] = {input.stride(0), input.stride(1), input.stride(2), input.stride(3)};
  const long long os[4] = {output.stride(0), output.stride(1), output.stride(2), output.stride(3)};
  const c10::cuda::CUDAGuard guard(input.device());
  raise(b200awq_rope_with_pos(input.data_ptr(), freqs.data_ptr<float>(), output.data_ptr(), s, b, h, d, d2, is, os, dt,
                              at::cuda::getCurrentCUDAStream().stream()),
        false);
  return output;
}

// reference: awq/kernels/csrc/position_embedding/pos_encoding_kernels.cu:56-88 (in place, returns nothing)
void rotary_embedding_neox(at::Tensor& positions, at::Tensor& query, at::Tensor& key, int head_size, at::Tensor& cos_sin_cache) {
  TORCH_CHECK(positions.is_cuda() && query.is_cuda() && key.is_cuda() && cos_sin_cache.is_cuda(), "all tensors must be CUDA tensors");
  TORCH_CHECK(positions.scalar_type() == at::ScalarType::Long && positions.is_contiguous(), "positions must be contiguous int64");
  const int dt = dtype_code(query, "rotary_embedding_neox");
  TORCH_CHECK(key.scalar_type() == query.scalar_type() && cos_sin_cache.scalar_type() == query.scalar_type(),
              "query, key and cos_sin_cache must have one dtype");
  TORCH_CHECK(query.is_contiguous() && key.is_contiguous() && cos_sin_cache.is_contiguous(), "tensors must be contiguous");
  TORCH_CHECK(query.dim() >= 3 && key.dim() >= 3 && cos_sin_cache.dim() == 2, "query / key [b, tokens, ..., heads, head_size]");
  TORCH_CHECK(query.size(-1) == head_size && key.size(-1) == head_size, "last dimension must be head_size");
  const int64_t tokens = query.size(0) * query.size(1);  // reference :63
  const int64_t q_heads = query.size(-2), k_heads = key.size(-2);
  const int64_t rot_dim = cos_sin_cache.size(1);         // reference :64
  TORCH_CHECK(query.numel() == tokens * q_heads * head_size && key.numel() == tokens * k_heads * head_size,
              "query / key must hold tokens x heads x head_size elements");
  TORCH_CHECK(positions.numel() >= tokens, "one position per token");
  const c10::cuda::CUDAGuard guard(query.device());
  raise(b200awq_rotary_embedding_neox(reinterpret_cast<const long long*>(positions.data_ptr<int64_t>()), query.data_ptr(),
                                      key.data_ptr(), cos_sin_cache.data_ptr(), (int)tokens, (int)q_heads, (int)k_heads,
                                      head_size, (int)rot_dim, q_heads * head_size, k_heads * head_size, dt,
                                      at::cuda::getCurrentCUDAStream().stream()),
        false);
}

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.doc() = "B200-native drop-in for llm-awq's awq_inference_engine (W4A16 path only)";
  m.def("gemm_forward_cuda_new", &gemm_forward_cuda_new, "New quantized GEMM kernel.");
  m.def("gemv_forward_cuda_new", &gemv_forward_cuda_new, "New quantized GEMV kernel.");
  m.def("layernorm_forward_cuda", &layernorm_forward_cuda, "FasterTransformer layernorm kernel");
  m.def("single_query_attention", &single_query_attention, "Attention with a single query", py::arg("q"), py::arg("k"),
        py::arg("v"), py::arg("k_cache"), py::arg("v_cache"), py::arg("length_per_sample_"), py::arg("alibi_slopes_"),
        py::arg("timestep"), py::arg("rotary_embedding_dim") = 0, py::arg("rotary_base") = 10000.0f,
        py::arg("rotary_scale") = 1.0f, py::arg("neox_rotary_style") = true);
  m.def("fused_rope_with_pos_forward_func", &fused_rope_with_pos_forward_func,
        "Fused rope forward function with B,S,D embedding");
  m.def("rotary_embedding_neox", &rotary_embedding_neox, "Apply GPT-NeoX style rotary embedding to query and key");
  m.def("mlp_front_forward_cuda", &mlp_front_forward_cuda, "silu(x Wgate^T) * (x Wup^T) for W4A16 weights, one call");
  m.def("set_pdl", [](bool on) { return b200awq_set_pdl(on ? 1 : 0) != 0; }, "programmatic dependent launch on/off");
  m.def("launch_count", []() { return b200awq_launch_count(); }, "kernels launched by libb200awq so far");
  m.def("version", []() { return std::string(b200awq_version()); });
}
