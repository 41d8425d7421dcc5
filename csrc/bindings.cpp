// Python bindings (torch extension `photon_b200._C`) for the sm_100a kernels in this directory.
// Tensors are passed as torch::Tensor; every op runs on the current CUDA stream of the tensor's device.
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <cuda_runtime.h>
#include <pybind11/pybind11.h>
#include <torch/extension.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <limits>
#include <string>
#include <vector>

#include "comm.h"
#include "decode.h"
#include "fp8_ops.h"
#include "fused_ops.h"
#include "gemm_tcgen05.h"
#include "attention_tcgen05.h"

namespace py = pybind11;
using torch::Tensor;

namespace {

std::atomic<long long> g_launches{0};

inline cudaStream_t stream_of(const Tensor& t) { return at::cuda::getCurrentCUDAStream(t.device().index()).stream(); }

inline void check_cuda(const Tensor& t, const char* name) {
  TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor");
}
inline void check_bf16(const Tensor& t, const char* name) {
  check_cuda(t, name);
  TORCH_CHECK(t.scalar_type() == at::kBFloat16, name, " must be bfloat16");
}
inline void check_f32(const Tensor& t, const char* name) {
  check_cuda(t, name);
  TORCH_CHECK(t.scalar_type() == at::kFloat, name, " must be float32");
}
inline const void* opt_ptr(const c10::optional<Tensor>& t) { return t.has_value() ? t->data_ptr() : nullptr; }

#define CUDA_OK(expr)                                                                        \
  do {                                                                                       \
    cudaError_t e__ = (expr);                                                                \
    TORCH_CHECK(e__ == cudaSuccess, #expr " failed: ", cudaGetErrorString(e__));             \
  } while (0)

// ---------------------------------------------------------------------------------- GEMM
// a: [M,K] (a_mn=0) or [K,M] (a_mn=1);  b: [N,K] (b_mn=0) or [K,N] (b_mn=1);  d: [M,N]
void gemm(const Tensor& a, const Tensor& b, Tensor& d, int a_mn, int b_mn, int epi, const c10::optional<Tensor>& bias,
          const c10::optional<Tensor>& aux, c10::optional<Tensor> d2, bool accumulate, double alpha, int cluster) {
  check_bf16(a, "a");
  check_bf16(b, "b");
  check_cuda(d, "d");
  TORCH_CHECK(a.dim() == 2 && b.dim() == 2 && d.dim() == 2, "gemm operands must be 2-D");
  TORCH_CHECK(a.stride(1) == 1 && b.stride(1) == 1 && d.stride(1) == 1, "gemm operands must have unit inner stride");
  c10::cuda::CUDAGuard guard(a.device());
  pb::GemmArgs g;
  g.M = int(a_mn ? a.size(1) : a.size(0));
  g.K = int(a_mn ? a.size(0) : a.size(1));
  g.N = int(b_mn ? b.size(1) : b.size(0));
  TORCH_CHECK((b_mn ? b.size(0) : b.size(1)) == g.K, "gemm: K mismatch between a and b");
  TORCH_CHECK(d.size(0) == g.M && d.size(1) == g.N, "gemm: output shape mismatch");
  g.A = a.data_ptr(), g.B = b.data_ptr(), g.D = d.data_ptr();
  g.lda = a.stride(0), g.ldb = b.stride(0), g.ldd = d.stride(0);
  g.a_mn = a_mn, g.b_mn = b_mn, g.epi = epi, g.accumulate = accumulate ? 1 : 0, g.alpha = float(alpha);
  if (epi == pb::EPI_F32) {
    TORCH_CHECK(d.scalar_type() == at::kFloat, "EPI_F32 needs a float32 output");
  } else {
    TORCH_CHECK(d.scalar_type() == at::kBFloat16, "bf16 epilogues need a bfloat16 output");
  }
  if (bias.has_value()) {
    check_f32(*bias, "bias");
    TORCH_CHECK(bias->numel() == g.N, "bias length must equal N");
    g.bias = bias->data_ptr<float>();
  }
  if (aux.has_value()) {
    check_bf16(*aux, "aux");
    TORCH_CHECK(aux->size(0) == g.M && aux->size(1) == g.N && aux->stride(1) == 1, "aux must be [M,N]");
    g.aux = aux->data_ptr(), g.ld_aux = aux->stride(0);
  }
  if (d2.has_value()) {
    check_bf16(*d2, "d2");
    TORCH_CHECK(d2->size(0) == g.M && d2->size(1) == g.N && d2->stride(1) == 1, "d2 must be [M,N]");
    g.D2 = d2->data_ptr(), g.ldd2 = d2->stride(0);
  }
  g.num_sms = at::cuda::getCurrentDeviceProperties()->multiProcessorCount;
  g.cluster = cluster;
  pb::gemm_bf16_launch(g, stream_of(a));
  g_launches += 1;
}

// fp8 operands (1-byte tensors: torch.uint8 or float8 storage). `meta` = float32 [3, n_roles] = (scale, scale_inv, amax) rows.
inline bool is_byte(const Tensor& t) {
  return t.scalar_type() == at::kByte || t.scalar_type() == at::kFloat8_e4m3fn || t.scalar_type() == at::kFloat8_e5m2;
}
void gemm_fp8(const Tensor& a, const Tensor& b, Tensor& d, int a_mn, int b_mn, int epi, int a_fmt, int b_fmt, const Tensor& meta, int role_a,
              int role_b, const c10::optional<Tensor>& bias, const c10::optional<Tensor>& aux, c10::optional<Tensor> d2, bool accumulate,
              double alpha, int cluster, c10::optional<Tensor> d8, int role_out) {
  check_cuda(a, "a");
  check_cuda(b, "b");
  check_cuda(d, "d");
  TORCH_CHECK(is_byte(a) && is_byte(b), "gemm_fp8 operands must be 1-byte tensors");
  TORCH_CHECK(a.dim() == 2 && b.dim() == 2 && d.dim() == 2, "gemm operands must be 2-D");
  TORCH_CHECK(a.stride(1) == 1 && b.stride(1) == 1 && d.stride(1) == 1, "gemm operands must have unit inner stride");
  check_f32(meta, "meta");
  TORCH_CHECK(meta.dim() == 2 && meta.size(0) == 3 && meta.is_contiguous(), "meta must be contiguous float32 [3, n_roles]");
  const int64_t nr = meta.size(1);
  TORCH_CHECK(role_a >= 0 && role_a < nr && role_b >= 0 && role_b < nr, "role index out of range");
  c10::cuda::CUDAGuard guard(a.device());
  pb::GemmArgs g;
  g.fp8 = 1, g.a_fmt = a_fmt, g.b_fmt = b_fmt;
  g.M = int(a_mn ? a.size(1) : a.size(0));
  g.K = int(a_mn ? a.size(0) : a.size(1));
  g.N = int(b_mn ? b.size(1) : b.size(0));
  TORCH_CHECK((b_mn ? b.size(0) : b.size(1)) == g.K, "gemm: K mismatch between a and b");
  TORCH_CHECK(d.size(0) == g.M && d.size(1) == g.N, "gemm: output shape mismatch");
  g.A = a.data_ptr(), g.B = b.data_ptr(), g.D = d.data_ptr();
  g.lda = a.stride(0), g.ldb = b.stride(0), g.ldd = d.stride(0);
  g.a_mn = a_mn, g.b_mn = b_mn, g.epi = epi, g.accumulate = accumulate ? 1 : 0, g.alpha = float(alpha);
  const float* m = meta.data_ptr<float>();
  g.sinv_a = m + nr + role_a, g.sinv_b = m + nr + role_b;
  if (epi == pb::EPI_F32) {
    TORCH_CHECK(d.scalar_type() == at::kFloat, "EPI_F32 needs a float32 output");
  } else {
    TORCH_CHECK(d.scalar_type() == at::kBFloat16, "bf16 epilogues need a bfloat16 output");
  }
  if (bias.has_value()) {
    check_f32(*bias, "bias");
    TORCH_CHECK(bias->numel() == g.N, "bias length must equal N");
    g.bias = bias->data_ptr<float>();
  }
  if (aux.has_value()) {
    check_bf16(*aux, "aux");
    TORCH_CHECK(aux->size(0) == g.M && aux->size(1) == g.N && aux->stride(1) == 1, "aux must be [M,N]");
    g.aux = aux->data_ptr(), g.ld_aux = aux->stride(0);
  }
  if (d2.has_value()) {
    check_bf16(*d2, "d2");
    TORCH_CHECK(d2->size(0) == g.M && d2->size(1) == g.N && d2->stride(1) == 1, "d2 must be [M,N]");
    g.D2 = d2->data_ptr(), g.ldd2 = d2->stride(0);
  }
  if (d8.has_value()) {
    TORCH_CHECK(is_byte(*d8) && d8->size(0) == g.M && d8->size(1) == g.N && d8->stride(1) == 1, "d8 must be a 1-byte [M,N] tensor");
    TORCH_CHECK(role_out >= 0 && role_out < nr, "role_out out of range");
    g.D8 = d8->data_ptr(), g.ldd8 = d8->stride(0);
    g.out_scale = m + role_out;
    g.out_amax = const_cast<float*>(m) + 2 * nr + role_out;
  }
  g.num_sms = at::cuda::getCurrentDeviceProperties()->multiProcessorCount;
  g.cluster = cluster;
  pb::gemm_launch(g, stream_of(a));
  g_launches += 1;
}
// block-scaled MXFP8: quantise a bf16 matrix (rows padded to `rblk` 128-row blocks in the scale array) / multiply
std::vector<Tensor> mx_quantize(const Tensor& x, int64_t rblk) {
  check_bf16(x, "x");
  TORCH_CHECK(x.dim() == 2 && x.stride(1) == 1 && x.size(1) % 128 == 0, "mx_quantize expects [R,K] with K a multiple of 128");
  const int64_t R = x.size(0), K = x.size(1);
  if (rblk <= 0) rblk = (R + 127) / 128;
  TORCH_CHECK(rblk * 128 >= R, "rblk too small");
  c10::cuda::CUDAGuard guard(x.device());
  auto q = torch::empty({R, K}, x.options().dtype(at::kByte));
  auto sf = torch::zeros({K / 128, rblk, 512}, x.options().dtype(at::kByte));
  pb::mx_quantize(x.data_ptr(), x.stride(0), q.data_ptr(), sf.data_ptr(), R, int(K), int(rblk), stream_of(x));
  g_launches += 1;
  return {q, sf};
}
void gemm_mxfp8(const Tensor& a8, const Tensor& b8, Tensor& d, const Tensor& sfa, const Tensor& sfb, const c10::optional<Tensor>& bias) {
  TORCH_CHECK(is_byte(a8) && is_byte(b8) && a8.is_contiguous() && b8.is_contiguous(), "gemm_mxfp8 operands must be contiguous 1-byte matrices");
  check_bf16(d, "d");
  const int M = int(a8.size(0)), K = int(a8.size(1)), N = int(b8.size(0));
  TORCH_CHECK(b8.size(1) == K && d.size(0) == M && d.size(1) == N && d.stride(1) == 1, "gemm_mxfp8: shape mismatch");
  TORCH_CHECK(sfa.is_contiguous() && sfa.numel() == int64_t(K / 128) * ((M + 127) / 128) * 512, "sfa must be [K/128][ceil(M/128)][512]");
  TORCH_CHECK(sfb.is_contiguous() && sfb.numel() == int64_t(K / 128) * (2 * ((N + 255) / 256)) * 512, "sfb must be [K/128][2*ceil(N/256)][512]");
  if (bias.has_value()) check_f32(*bias, "bias");
  c10::cuda::CUDAGuard guard(a8.device());
  pb::gemm_mxfp8_launch(a8.data_ptr(), b8.data_ptr(), d.data_ptr(), sfa.data_ptr(), sfb.data_ptr(),
                        bias.has_value() ? bias->data_ptr<float>() : nullptr, M, N, K, d.stride(0),
                        at::cuda::getCurrentDeviceProperties()->multiProcessorCount, stream_of(a8));
  g_launches += 1;
}
void layernorm_fwd_q8(const Tensor& x, const Tensor& gamma, const c10::optional<Tensor>& beta, Tensor& y8, Tensor& mean, Tensor& rstd,
                      double eps, Tensor& meta, int role) {
  check_bf16(x, "x");
  check_f32(gamma, "gamma");
  check_f32(meta, "meta");
  TORCH_CHECK(x.is_contiguous() && y8.is_contiguous() && is_byte(y8) && y8.numel() == x.numel(), "layernorm_fwd_q8: y8 must be a contiguous 1-byte tensor shaped like x");
  const int64_t nr = meta.size(1);
  TORCH_CHECK(meta.dim() == 2 && meta.size(0) == 3 && role >= 0 && role < nr, "bad meta / role");
  c10::cuda::CUDAGuard guard(x.device());
  const int d = int(x.size(-1));
  float* m = meta.data_ptr<float>();
  pb::layernorm_fwd_q8(x.data_ptr(), gamma.data_ptr<float>(), beta.has_value() ? beta->data_ptr<float>() : nullptr, y8.data_ptr(),
                       mean.data_ptr<float>(), rstd.data_ptr<float>(), x.numel() / d, d, float(eps), m + role, m + 2 * nr + role, stream_of(x));
  g_launches += 1;
}
// out_sum[j] += sum_t dy[t,j] and / or y8 = fp8(dy * scale[role]) with amax[role] updated — one read of dy
void colsum_quant(const Tensor& dy, c10::optional<Tensor> out_sum, c10::optional<Tensor> y8, int fmt, c10::optional<Tensor> meta, int role) {
  check_bf16(dy, "dy");
  TORCH_CHECK(dy.dim() == 2 && dy.stride(1) == 1, "colsum_quant expects [T,N] with unit inner stride");
  c10::cuda::CUDAGuard guard(dy.device());
  const float* scale = nullptr;
  float* amax = nullptr;
  void* y = nullptr;
  long long ld8 = 0;
  if (y8.has_value()) {
    TORCH_CHECK(meta.has_value(), "quantising needs the meta tensor");
    check_f32(*meta, "meta");
    const int64_t nr = meta->size(1);
    TORCH_CHECK(meta->dim() == 2 && meta->size(0) == 3 && role >= 0 && role < nr, "bad meta / role");
    TORCH_CHECK(is_byte(*y8) && y8->dim() == 2 && y8->size(0) == dy.size(0) && y8->size(1) == dy.size(1) && y8->stride(1) == 1 &&
                    y8->stride(0) % 8 == 0, "y8 must be a 1-byte [T,N] tensor");
    scale = meta->data_ptr<float>() + role;
    amax = meta->data_ptr<float>() + 2 * nr + role;
    y = y8->data_ptr(), ld8 = y8->stride(0);
  }
  if (out_sum.has_value()) check_f32(*out_sum, "out_sum");
  pb::colsum_quant(dy.data_ptr(), dy.stride(0), out_sum.has_value() ? out_sum->data_ptr<float>() : nullptr, y, ld8, fmt, scale, amax,
                   dy.size(0), int(dy.size(1)), stream_of(dy));
  g_launches += 1;
}
void fp8_quantize_segments(const Tensor& src, Tensor& dst8, const Tensor& seg, Tensor& meta, int role0) {
  check_bf16(src, "src");
  check_cuda(seg, "seg");
  check_f32(meta, "meta");
  TORCH_CHECK(seg.scalar_type() == at::kLong && seg.dim() == 2 && seg.size(1) == 2 && seg.is_contiguous(), "seg must be int64 [n,2] on the device");
  TORCH_CHECK(is_byte(dst8) && dst8.numel() >= src.numel(), "dst8 must be a 1-byte tensor at least as long as src");
  const int64_t nr = meta.size(1);
  const int n = int(seg.size(0));
  TORCH_CHECK(role0 >= 0 && role0 + n <= nr, "roles out of range");
  c10::cuda::CUDAGuard guard(src.device());
  float* m = meta.data_ptr<float>();
  pb::quantize_segments(src.data_ptr(), dst8.data_ptr(), reinterpret_cast<const long long*>(seg.data_ptr<int64_t>()), n, m + role0,
                        m + nr + role0, m + 2 * nr + role0, stream_of(src));
  g_launches += 2;
}
void fp8_update_scales(Tensor& meta, Tensor& hist, const Tensor& fmax, Tensor& pos, int n, double margin_mult) {
  check_f32(meta, "meta");
  check_f32(hist, "hist");
  check_f32(fmax, "fmax");
  TORCH_CHECK(pos.scalar_type() == at::kInt && pos.is_cuda(), "pos must be an int32 device tensor");
  const int64_t nr = meta.size(1);
  TORCH_CHECK(n <= nr && hist.dim() == 2 && hist.size(0) >= n && fmax.numel() >= n && hist.is_contiguous(), "bad history / fmax shapes");
  c10::cuda::CUDAGuard guard(meta.device());
  float* m = meta.data_ptr<float>();
  pb::update_scales(m, m + nr, m + 2 * nr, hist.data_ptr<float>(), fmax.data_ptr<float>(), pos.data_ptr<int>(), n, int(hist.size(1)),
                    float(margin_mult), stream_of(meta));
  g_launches += 1;
}

// ---------------------------------------------------------------------------------- attention
void attention_fwd(const Tensor& qkv, Tensor& out, Tensor& lse, int n_heads, double scale, bool causal,
                   const c10::optional<Tensor>& alibi_slopes) {
  check_bf16(qkv, "qkv");
  check_bf16(out, "out");
  check_f32(lse, "lse");
  TORCH_CHECK(qkv.dim() == 3 && qkv.is_contiguous(), "qkv must be contiguous [B,S,3*d]");
  c10::cuda::CUDAGuard guard(qkv.device());
  const int B = int(qkv.size(0)), S = int(qkv.size(1)), d = int(qkv.size(2) / 3);
  if (alibi_slopes.has_value()) {
    check_f32(*alibi_slopes, "alibi_slopes");
    TORCH_CHECK(alibi_slopes->numel() == n_heads, "alibi_slopes must have n_heads elements");
  }
  pb::attention_fwd_launch(qkv.data_ptr(), out.data_ptr(), lse.data_ptr<float>(), B, S, n_heads, d / n_heads, float(scale), causal,
                           at::cuda::getCurrentDeviceProperties()->multiProcessorCount, stream_of(qkv),
                           alibi_slopes.has_value() ? alibi_slopes->data_ptr<float>() : nullptr);
  g_launches += 1;
}
void attention_bwd(const Tensor& qkv, const Tensor& out, const Tensor& dout, const Tensor& lse, Tensor& dqkv, Tensor& delta,
                   int n_heads, double scale, bool causal, const c10::optional<Tensor>& alibi_slopes) {
  check_bf16(qkv, "qkv");
  check_bf16(out, "out");
  check_bf16(dout, "dout");
  check_bf16(dqkv, "dqkv");
  check_f32(lse, "lse");
  check_f32(delta, "delta");
  c10::cuda::CUDAGuard guard(qkv.device());
  const int B = int(qkv.size(0)), S = int(qkv.size(1)), d = int(qkv.size(2) / 3);
  const int launched = pb::attention_bwd_launch(qkv.data_ptr(), out.data_ptr(), dout.data_ptr(), lse.data_ptr<float>(), dqkv.data_ptr(),
                                                delta.data_ptr<float>(), B, S, n_heads, d / n_heads, float(scale), causal,
                                                at::cuda::getCurrentDeviceProperties()->multiProcessorCount, stream_of(qkv),
                                                alibi_slopes.has_value() ? alibi_slopes->data_ptr<float>() : nullptr);
  g_launches += launched;
}
void rope(Tensor& qkv, const Tensor& cos_t, const Tensor& sin_t, int n_heads, bool inverse) {
  check_bf16(qkv, "qkv");
  check_f32(cos_t, "cos");
  check_f32(sin_t, "sin");
  TORCH_CHECK(qkv.dim() == 3 && qkv.is_contiguous(), "qkv must be contiguous [B,S,3*d]");
  c10::cuda::CUDAGuard guard(qkv.device());
  const int S = int(qkv.size(1)), d = int(qkv.size(2) / 3), dh = d / n_heads;
  TORCH_CHECK(cos_t.is_contiguous() && sin_t.is_contiguous() && cos_t.size(0) >= S && cos_t.size(1) == dh / 2, "cos/sin must be [>=S, dh/2]");
  pb::rope_launch(qkv.data_ptr(), cos_t.data_ptr<float>(), sin_t.data_ptr<float>(), (long long)qkv.size(0) * S, S, n_heads, dh, inverse,
                  stream_of(qkv));
  g_launches += 1;
}

// ---------------------------------------------------------------------------------- fused ops
void embed_fwd(const Tensor& ids, const Tensor& wte, const c10::optional<Tensor>& wpe, Tensor& out, int S) {
  check_cuda(ids, "ids");
  TORCH_CHECK(ids.scalar_type() == at::kLong && ids.is_contiguous(), "ids must be contiguous int64");
  check_bf16(wte, "wte");
  check_bf16(out, "out");
  c10::cuda::CUDAGuard guard(ids.device());
  pb::embed_fwd(ids.data_ptr<int64_t>(), wte.data_ptr(), opt_ptr(wpe), out.data_ptr(), ids.numel(), S, int(wte.size(1)),
                int(wte.size(0)), stream_of(ids));
  g_launches += 1;
}
void embed_bwd(const Tensor& ids, const Tensor& dh, Tensor& dwte, c10::optional<Tensor> dwpe, int S) {
  check_bf16(dh, "dh");
  check_f32(dwte, "dwte");
  c10::cuda::CUDAGuard guard(ids.device());
  pb::embed_bwd(ids.data_ptr<int64_t>(), dh.data_ptr(), dwte.data_ptr<float>(), dwpe.has_value() ? dwpe->data_ptr<float>() : nullptr,
                ids.numel(), S, int(dwte.size(1)), int(dwte.size(0)), stream_of(ids));
  g_launches += dwpe.has_value() ? 2 : 1;
}
void layernorm_fwd(const Tensor& x, const Tensor& gamma, const c10::optional<Tensor>& beta, Tensor& y, Tensor& mean, Tensor& rstd,
                   double eps) {
  check_bf16(x, "x");
  check_f32(gamma, "gamma");
  TORCH_CHECK(x.is_contiguous() && y.is_contiguous(), "layernorm tensors must be contiguous");
  c10::cuda::CUDAGuard guard(x.device());
  const int d = int(x.size(-1));
  pb::layernorm_fwd(x.data_ptr(), gamma.data_ptr<float>(), beta.has_value() ? beta->data_ptr<float>() : nullptr, y.data_ptr(),
                    mean.data_ptr<float>(), rstd.data_ptr<float>(), x.numel() / d, d, float(eps), stream_of(x));
  g_launches += 1;
}
void layernorm_bwd(const Tensor& dy, const Tensor& x, const Tensor& gamma, const Tensor& mean, const Tensor& rstd,
                   const c10::optional<Tensor>& dres, Tensor& dx, c10::optional<Tensor> dgamma, c10::optional<Tensor> dbeta) {
  check_bf16(dy, "dy");
  check_bf16(x, "x");
  TORCH_CHECK(dy.is_contiguous() && x.is_contiguous() && dx.is_contiguous(), "layernorm tensors must be contiguous");
  c10::cuda::CUDAGuard guard(x.device());
  const int d = int(x.size(-1));
  pb::layernorm_bwd(dy.data_ptr(), x.data_ptr(), gamma.data_ptr<float>(), mean.data_ptr<float>(), rstd.data_ptr<float>(), opt_ptr(dres),
                    dx.data_ptr(), dgamma.has_value() ? dgamma->data_ptr<float>() : nullptr,
                    dbeta.has_value() ? dbeta->data_ptr<float>() : nullptr, x.numel() / d, d, stream_of(x));
  g_launches += (dgamma.has_value() || dbeta.has_value()) ? 2 : 1;
}
void col_sum(const Tensor& dy, Tensor& out) {
  check_bf16(dy, "dy");
  check_f32(out, "out");
  TORCH_CHECK(dy.dim() == 2 && dy.stride(1) == 1, "col_sum expects [T,N] with unit inner stride");
  c10::cuda::CUDAGuard guard(dy.device());
  pb::col_reduce(dy.data_ptr(), dy.stride(0), nullptr, nullptr, nullptr, out.data_ptr<float>(), nullptr, dy.size(0), int(dy.size(1)),
                 stream_of(dy));
  g_launches += 1;
}
void cross_entropy(Tensor& logits, const Tensor& targets, double grad_scale, bool write_grad, Tensor& stats,
                   c10::optional<Tensor> row_lse, const c10::optional<Tensor>& unigram_logp) {
  check_bf16(logits, "logits");
  TORCH_CHECK(logits.dim() == 2 && logits.stride(1) == 1, "logits must be [rows,V]");
  TORCH_CHECK(targets.scalar_type() == at::kLong && targets.is_contiguous(), "targets must be contiguous int64");
  TORCH_CHECK(stats.scalar_type() == at::kDouble && stats.numel() >= 4, "stats must be float64[>=4]");
  c10::cuda::CUDAGuard guard(logits.device());
  pb::cross_entropy(logits.data_ptr(), logits.stride(0), targets.data_ptr<int64_t>(), logits.size(0), int(logits.size(1)), float(grad_scale),
                    write_grad, stats.data_ptr<double>(), row_lse.has_value() ? row_lse->data_ptr<float>() : nullptr,
                    unigram_logp.has_value() ? unigram_logp->data_ptr<float>() : nullptr, stream_of(logits));
  g_launches += 1;
}
void flat_l2_norm(const Tensor& x, Tensor& scratch_f64, Tensor& out_f32) {
  check_f32(x, "x");
  c10::cuda::CUDAGuard guard(x.device());
  cudaStream_t st = stream_of(x);
  CUDA_OK(cudaMemsetAsync(scratch_f64.data_ptr(), 0, sizeof(double), st));
  pb::flat_sqnorm(x.data_ptr<float>(), x.numel(), scratch_f64.data_ptr<double>(), st);
  pb::sqrt_finalize(scratch_f64.data_ptr<double>(), out_f32.data_ptr<float>(), st);
  g_launches += 2;
}
void axpby(Tensor& acc, const Tensor& x, double a, double b) {
  check_f32(acc, "acc");
  check_f32(x, "x");
  TORCH_CHECK(acc.numel() == x.numel() && acc.numel() % 4 == 0, "axpby: sizes must match and be multiples of 4");
  c10::cuda::CUDAGuard guard(acc.device());
  pb::axpby(acc.data_ptr<float>(), x.data_ptr<float>(), float(a), float(b), acc.numel(), stream_of(acc));
  g_launches += 1;
}
void cast_bf16(const Tensor& src, Tensor& dst) {
  check_f32(src, "src");
  check_bf16(dst, "dst");
  TORCH_CHECK(src.numel() == dst.numel() && src.numel() % 4 == 0, "cast: sizes must match and be multiples of 4");
  c10::cuda::CUDAGuard guard(src.device());
  pb::cast_fp32_to_bf16(src.data_ptr<float>(), dst.data_ptr(), src.numel(), stream_of(src));
  g_launches += 1;
}
void fused_optimizer(Tensor& p, const Tensor& g, Tensor& m, Tensor& v, c10::optional<Tensor> shadow, int kind, bool first_step, double lr,
                     double beta1, double beta2, double eps, double decay, double clip, double step_size, double inv_sqrt_bc2,
                     const c10::optional<Tensor>& grad_mult) {
  check_f32(p, "p");
  check_f32(g, "g");
  TORCH_CHECK(p.numel() % 4 == 0, "flat buffers must be multiples of 4 elements");
  c10::cuda::CUDAGuard guard(p.device());
  pb::OptimHyper h;
  h.kind = kind, h.first_step = first_step ? 1 : 0;
  h.lr = float(lr), h.beta1 = float(beta1), h.beta2 = float(beta2), h.eps = float(eps), h.decay = float(decay);
  h.clip = std::isfinite(clip) ? float(clip) : std::numeric_limits<float>::infinity();
  h.step_size = float(step_size), h.inv_sqrt_bc2 = float(inv_sqrt_bc2);
  pb::fused_optimizer(p.data_ptr<float>(), g.data_ptr<float>(), m.data_ptr<float>(), v.data_ptr<float>(),
                      shadow.has_value() ? shadow->data_ptr() : nullptr, p.numel(), h,
                      grad_mult.has_value() ? grad_mult->data_ptr<float>() : nullptr, stream_of(p));
  g_launches += 1;
}

// ---------------------------------------------------------------------------------- KV-cached decoding
inline void check_i32(const Tensor& t, const char* name, int64_t n) {
  check_cuda(t, name);
  TORCH_CHECK(t.scalar_type() == at::kInt && t.is_contiguous() && t.numel() == n, name, " must be a contiguous int32 tensor of ", n,
              " elements");
}
// embedding rows at explicit positions: out[t] = wte[ids[t]] (+ wpe[pos[t]])
void embed_at(const Tensor& ids, const Tensor& pos, const Tensor& wte, const c10::optional<Tensor>& wpe, Tensor& out) {
  check_cuda(ids, "ids");
  TORCH_CHECK(ids.scalar_type() == at::kLong && ids.is_contiguous(), "ids must be contiguous int64");
  check_i32(pos, "pos", ids.numel());
  check_bf16(wte, "wte");
  check_bf16(out, "out");
  const int64_t d = wte.size(1);
  TORCH_CHECK(out.is_contiguous() && out.numel() == ids.numel() * d, "out must be contiguous [T, d]");
  if (wpe.has_value()) {
    check_bf16(*wpe, "wpe");
    TORCH_CHECK(wpe->dim() == 2 && wpe->size(1) == d, "wpe must be [max_pos, d]");
  }
  c10::cuda::CUDAGuard guard(ids.device());
  pb::embed_fwd(ids.data_ptr<int64_t>(), wte.data_ptr(), opt_ptr(wpe), out.data_ptr(), ids.numel(), wpe.has_value() ? int(wpe->size(0)) : 1,
                int(d), int(wte.size(0)), stream_of(ids), pos.data_ptr<int>());
  g_launches += 1;
}
int64_t decode_attention_splits(int64_t BH, int64_t s_max) {
  return pb::decode_attention_splits(int(BH), int(s_max), at::cuda::getCurrentDeviceProperties()->multiProcessorCount);
}
// q: [B, >= d] rows (row stride ldq, e.g. the q third of qkv [B, 3d]); kv: [B, S_max, 2d]; lengths int32 [B]; out [B, d]
void decode_attention(const Tensor& q, const Tensor& kv, const Tensor& lengths, const c10::optional<Tensor>& alibi_slopes, double scale,
                      int n_heads, int n_split, Tensor& out, c10::optional<Tensor> lse) {
  check_bf16(q, "q");
  check_bf16(kv, "kv");
  check_bf16(out, "out");
  TORCH_CHECK(kv.dim() == 3 && kv.is_contiguous(), "kv must be a contiguous [B, S_max, 2d] cache");
  const int B = int(kv.size(0)), S = int(kv.size(1)), d = int(kv.size(2) / 2);
  TORCH_CHECK(n_heads > 0 && d % n_heads == 0, "d must be a multiple of n_heads");
  const int dh = d / n_heads;
  TORCH_CHECK(dh == 64 || dh == 128, "decode_attention covers d_head 64 and 128");
  TORCH_CHECK(q.dim() == 2 && q.size(0) == B && q.size(1) >= d && q.stride(1) == 1 && q.stride(0) % 8 == 0, "q must be [B, >= d] rows");
  TORCH_CHECK(out.dim() == 2 && out.size(0) == B && out.size(1) == d && out.is_contiguous(), "out must be contiguous [B, d]");
  check_i32(lengths, "lengths", B);
  if (alibi_slopes.has_value()) {
    check_f32(*alibi_slopes, "alibi_slopes");
    TORCH_CHECK(alibi_slopes->numel() == n_heads && alibi_slopes->is_contiguous(), "alibi_slopes must have n_heads elements");
  }
  if (lse.has_value()) {
    check_f32(*lse, "lse");
    TORCH_CHECK(lse->is_contiguous() && lse->numel() == int64_t(B) * n_heads, "lse must be contiguous [B, H]");
  }
  c10::cuda::CUDAGuard guard(q.device());
  const int max_split = (S + pb::DECODE_TILE_KEYS - 1) / pb::DECODE_TILE_KEYS;
  if (n_split <= 0) n_split = pb::decode_attention_splits(B * n_heads, S, at::cuda::getCurrentDeviceProperties()->multiProcessorCount);
  TORCH_CHECK(n_split <= std::max(max_split, 1), "n_split must be <= ceil(S_max / ", pb::DECODE_TILE_KEYS, ")");
  Tensor scratch;
  if (n_split > 1) scratch = torch::empty({int64_t(B) * n_heads * n_split * (dh + 2)}, q.options().dtype(at::kFloat));
  g_launches += pb::decode_attention_launch(q.data_ptr(), q.stride(0), kv.data_ptr(), B, S, n_heads, dh, lengths.data_ptr<int>(),
                                            alibi_slopes.has_value() ? alibi_slopes->data_ptr<float>() : nullptr, float(scale), n_split,
                                            n_split > 1 ? scratch.data_ptr<float>() : nullptr, out.data_ptr(),
                                            lse.has_value() ? lse->data_ptr<float>() : nullptr, stream_of(q));
}
// cache[b_idx[t], pos[t]] = k|v of qkv row t (after RoPE of q and k at pos[t] when cos / sin are given)
void kv_write(Tensor& qkv, Tensor& cache, const Tensor& b_idx, const Tensor& pos, const c10::optional<Tensor>& cos_t,
              const c10::optional<Tensor>& sin_t, int n_heads) {
  check_bf16(qkv, "qkv");
  check_bf16(cache, "cache");
  TORCH_CHECK(qkv.dim() == 2 && qkv.is_contiguous(), "qkv must be contiguous [T, 3d]");
  TORCH_CHECK(cache.dim() == 3 && cache.is_contiguous() && cache.size(2) * 3 == qkv.size(1) * 2, "cache must be contiguous [B, S_max, 2d]");
  const int64_t T = qkv.size(0);
  const int d = int(qkv.size(1) / 3);
  TORCH_CHECK(n_heads > 0 && d % n_heads == 0, "d must be a multiple of n_heads");
  const int dh = d / n_heads;
  check_i32(b_idx, "b_idx", T);
  check_i32(pos, "pos", T);
  const bool rotate = cos_t.has_value();
  TORCH_CHECK(rotate == sin_t.has_value(), "cos and sin go together");
  if (rotate) {
    check_f32(*cos_t, "cos");
    check_f32(*sin_t, "sin");
    TORCH_CHECK(cos_t->is_contiguous() && sin_t->is_contiguous() && cos_t->size(0) >= cache.size(1) && cos_t->size(1) == dh / 2 &&
                    sin_t->sizes() == cos_t->sizes(), "cos/sin must be [>= S_max, dh/2]");
  }
  c10::cuda::CUDAGuard guard(qkv.device());
  pb::kv_write_launch(qkv.data_ptr(), qkv.stride(0), cache.data_ptr(), int(cache.size(0)), int(cache.size(1)), b_idx.data_ptr<int>(),
                      pos.data_ptr<int>(), rotate ? cos_t->data_ptr<float>() : nullptr, rotate ? sin_t->data_ptr<float>() : nullptr, T,
                      n_heads, dh, rotate, stream_of(qkv));
  g_launches += 1;
}
void argmax_rows(const Tensor& logits, Tensor& out) {
  check_bf16(logits, "logits");
  TORCH_CHECK(logits.dim() == 2 && logits.stride(1) == 1, "logits must be [R, V] with unit inner stride");
  check_cuda(out, "out");
  TORCH_CHECK(out.scalar_type() == at::kLong && out.is_contiguous() && out.numel() == logits.size(0), "out must be contiguous int64 [R]");
  c10::cuda::CUDAGuard guard(logits.device());
  pb::argmax_rows_launch(logits.data_ptr(), logits.stride(0), logits.size(0), int(logits.size(1)), out.data_ptr<int64_t>(), stream_of(logits));
  g_launches += 1;
}

// ---------------------------------------------------------------------------------- symmetric arena (CUDA IPC)
int64_t ipc_alloc(int64_t nbytes, int device) {
  c10::cuda::CUDAGuard guard(static_cast<c10::DeviceIndex>(device));
  void* p = nullptr;
  CUDA_OK(cudaMalloc(&p, size_t(nbytes)));
  CUDA_OK(cudaMemset(p, 0, size_t(nbytes)));
  return reinterpret_cast<int64_t>(p);
}
py::bytes ipc_get_handle(int64_t ptr) {
  cudaIpcMemHandle_t h;
  CUDA_OK(cudaIpcGetMemHandle(&h, reinterpret_cast<void*>(ptr)));
  return py::bytes(reinterpret_cast<const char*>(&h), sizeof(h));
}
int64_t ipc_open_handle(const std::string& handle, int device) {
  c10::cuda::CUDAGuard guard(static_cast<c10::DeviceIndex>(device));
  TORCH_CHECK(handle.size() == sizeof(cudaIpcMemHandle_t), "bad IPC handle size");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle.data(), sizeof(h));
  void* p = nullptr;
  CUDA_OK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
  return reinterpret_cast<int64_t>(p);
}
void ipc_close(int64_t ptr) { CUDA_OK(cudaIpcCloseMemHandle(reinterpret_cast<void*>(ptr))); }
void ipc_free(int64_t ptr) { CUDA_OK(cudaFree(reinterpret_cast<void*>(ptr))); }
bool enable_peer_access(int device, int peer) {
  c10::cuda::CUDAGuard guard(static_cast<c10::DeviceIndex>(device));
  int can = 0;
  CUDA_OK(cudaDeviceCanAccessPeer(&can, device, peer));
  if (!can) return false;
  cudaError_t e = cudaDeviceEnablePeerAccess(peer, 0);
  if (e == cudaErrorPeerAccessAlreadyEnabled) {
    cudaGetLastError();
    return true;
  }
  CUDA_OK(e);
  return true;
}
Tensor tensor_from_ptr(int64_t ptr, int64_t numel, const std::string& dtype, int device) {
  auto dt = dtype == "float32" ? at::kFloat : dtype == "bfloat16" ? at::kBFloat16 : dtype == "int32" ? at::kInt
          : dtype == "float64" ? at::kDouble : at::kByte;
  auto opts = torch::TensorOptions().dtype(dt).device(torch::kCUDA, device);
  return torch::from_blob(reinterpret_cast<void*>(ptr), {numel}, [](void*) {}, opts);
}

std::atomic<long long> g_comm_timeout_ms{120000};   // bound on every cross-GPU spin inside the NVLink kernels (0 = forever)

pb::CommCtl make_ctl(const std::vector<int64_t>& ctl_ptrs, int rank) {
  TORCH_CHECK(ctl_ptrs.size() >= 1 && ctl_ptrs.size() <= pb::MAX_PEERS, "1..8 peers supported");
  pb::CommCtl c{};
  c.n = int(ctl_ptrs.size());
  c.rank = rank;
  c.timeout_ns = static_cast<unsigned long long>(g_comm_timeout_ms.load()) * 1000000ull;
  for (int i = 0; i < c.n; ++i) c.ctl[i] = reinterpret_cast<uint32_t*>(ctl_ptrs[i]);
  return c;
}

void fed_round(const std::vector<int64_t>& ctl_ptrs, int rank, int device, int64_t epoch, const std::vector<int64_t>& acc_ptrs,
               const std::vector<int64_t>& xg_ptrs, const std::vector<int64_t>& xs_ptrs, int64_t m_ptr, int64_t v_ptr, int64_t lo, int64_t hi, int64_t total,
               int kind, double avg_scale, double lr, double mu, double eta, double beta1, double beta2, double tau, int64_t round_t,
               bool sign_compat, int64_t acc_mc, int64_t xg_mc, const c10::optional<Tensor>& seg_bounds, c10::optional<Tensor> seg_sums,
               double wsum, bool zero_seg_sums) {
  c10::cuda::CUDAGuard guard(static_cast<c10::DeviceIndex>(device));
  pb::CommCtl c = make_ctl(ctl_ptrs, rank);
  pb::FedRoundArgs a{};
  for (int i = 0; i < c.n; ++i) {
    a.acc[i] = reinterpret_cast<const float*>(acc_ptrs[i]);
    a.xg[i] = reinterpret_cast<float*>(xg_ptrs[i]);
    a.xs[i] = xs_ptrs.empty() ? nullptr : reinterpret_cast<void*>(xs_ptrs[i]);
  }
  a.x = a.xg[rank];
  a.m = reinterpret_cast<float*>(m_ptr);
  a.v = reinterpret_cast<float*>(v_ptr);
  a.lo = lo, a.hi = hi, a.total = total, a.kind = kind, a.avg_scale = float(avg_scale), a.lr = float(lr), a.mu = float(mu);
  a.eta = float(eta), a.beta1 = float(beta1), a.beta2 = float(beta2), a.tau = float(tau);
  const double t = double(round_t < 1 ? 1 : round_t);
  a.inv_bc1 = float(1.0 / (1.0 - std::pow(beta1, t)));
  a.inv_bc2 = float(1.0 / (1.0 - std::pow(beta2, t)));
  a.sign = sign_compat ? 1.0f : -1.0f;
  a.acc_mc = reinterpret_cast<const float*>(acc_mc);   // NVLS multicast addresses (0 = P2P loops)
  a.xg_mc = reinterpret_cast<float*>(xg_mc);
  a.publish_wsum = wsum >= 0.0 ? 1 : 0;        // negative = the page was filled by set_wsum before (legacy callers)
  a.wsum = float(wsum >= 0.0 ? wsum : 0.0);
  a.zero_seg_sums = zero_seg_sums ? 1 : 0;
  {
    static const int walk = [] { const char* e = std::getenv("PB_ROUND_WALK"); return e ? std::atoi(e) : 0; }();
    a.walk = walk;
  }
  if (seg_bounds.has_value() && seg_sums.has_value()) {
    TORCH_CHECK(seg_bounds->is_cuda() && seg_bounds->scalar_type() == at::kLong && seg_bounds->is_contiguous() && seg_bounds->numel() >= 2,
                "seg_bounds must be a contiguous int64 device tensor with n_seg + 1 entries");
    a.n_seg = int(seg_bounds->numel()) - 1;
    TORCH_CHECK(seg_sums->is_cuda() && seg_sums->scalar_type() == at::kDouble && seg_sums->is_contiguous() && seg_sums->numel() == 5 * a.n_seg,
                "seg_sums must be a contiguous float64 device tensor [5, n_seg]");
    a.seg_bounds = reinterpret_cast<const long long*>(seg_bounds->data_ptr<int64_t>());
    a.seg_sums = seg_sums->data_ptr<double>();
  }
  pb::fed_round_launch(a, c, uint32_t(epoch), at::cuda::getCurrentDeviceProperties()->multiProcessorCount,
                       at::cuda::getCurrentCUDAStream(device).stream());
  g_launches += 1;
}
// ZeRO-3: accumulate the mean over ranks of slice `rank` of the unit's staging planes into `dst` (see comm.cu)
void zero3_reduce(const std::vector<int64_t>& ctl_ptrs, int rank, int device, int64_t epoch, const std::vector<int64_t>& stage_ptrs,
                  int64_t stage_mc, c10::optional<Tensor> dst, int64_t per) {
  c10::cuda::CUDAGuard guard(static_cast<c10::DeviceIndex>(device));
  pb::CommCtl c = make_ctl(ctl_ptrs, rank);
  pb::ShardReduceArgs a{};
  TORCH_CHECK(per % 4 == 0 && per >= 0, "slice length must be a multiple of 4");
  if (per > 0) {
    TORCH_CHECK(dst.has_value() && dst->scalar_type() == at::kFloat && dst->numel() >= per && dst->is_contiguous(), "dst: fp32, >= per");
    TORCH_CHECK(int(stage_ptrs.size()) == c.n, "one staging plane per rank");
    for (int i = 0; i < c.n; ++i) a.stage[i] = reinterpret_cast<const float*>(stage_ptrs[i]);
    a.dst = dst->data_ptr<float>();
  }
  a.stage_mc = reinterpret_cast<const float*>(stage_mc);
  a.per = per;
  a.scale = 1.0f / float(c.n);
  pb::zero3_reduce_launch(a, c, uint32_t(epoch), at::cuda::getCurrentDeviceProperties()->multiProcessorCount,
                          at::cuda::getCurrentCUDAStream(device).stream());
  g_launches += 1;
}

// device-to-device copy between (possibly peer-mapped) raw addresses on the current stream: the copy engines pull a parameter
// slice from its owner over NVLink without occupying an SM
void memcpy_async(int64_t dst, int64_t src, int64_t nbytes, int device) {
  c10::cuda::CUDAGuard guard(static_cast<c10::DeviceIndex>(device));
  cudaError_t e = cudaMemcpyAsync(reinterpret_cast<void*>(dst), reinterpret_cast<const void*>(src), size_t(nbytes), cudaMemcpyDefault,
                                  at::cuda::getCurrentCUDAStream(device).stream());
  TORCH_CHECK(e == cudaSuccess, "memcpy_async: ", cudaGetErrorString(e));
}

void ddp_allreduce(const std::vector<int64_t>& ctl_ptrs, int rank, int device, int64_t epoch, const std::vector<int64_t>& buf_ptrs, int64_t lo,
                   int64_t hi, c10::optional<Tensor> out_norm, int64_t buf_mc) {
  c10::cuda::CUDAGuard guard(static_cast<c10::DeviceIndex>(device));
  pb::CommCtl c = make_ctl(ctl_ptrs, rank);
  pb::AllReduceArgs a{};
  for (int i = 0; i < c.n; ++i) a.buf[i] = reinterpret_cast<float*>(buf_ptrs[i]);
  a.lo = lo, a.hi = hi;
  a.buf_mc = reinterpret_cast<float*>(buf_mc);
  pb::ddp_allreduce_launch(a, c, uint32_t(epoch), out_norm.has_value() ? out_norm->data_ptr<float>() : nullptr,
                           at::cuda::getCurrentDeviceProperties()->multiProcessorCount, at::cuda::getCurrentCUDAStream(device).stream());
  g_launches += out_norm.has_value() ? 2 : 1;
}
void ddp_zero_step(const std::vector<int64_t>& ctl_ptrs, int rank, int device, int64_t epoch, const std::vector<int64_t>& grad_ptrs,
                   const std::vector<int64_t>& param_ptrs, const std::vector<int64_t>& shadow_ptrs, Tensor m, Tensor v, int64_t lo, int64_t hi,
                   int64_t kind, bool first_step, double lr, double beta1, double beta2, double eps, double decay, double clip,
                   double step_size, double inv_sqrt_bc2, double max_norm, double grad_mult, c10::optional<Tensor> out_norm,
                   int64_t grads_mc, int64_t params_mc, int64_t shadow_mc) {
  c10::cuda::CUDAGuard guard(static_cast<c10::DeviceIndex>(device));
  pb::CommCtl c = make_ctl(ctl_ptrs, rank);
  pb::ZeroStepArgs a{};
  for (int i = 0; i < c.n; ++i) {
    a.grads[i] = reinterpret_cast<float*>(grad_ptrs[i]);
    a.params[i] = reinterpret_cast<float*>(param_ptrs[i]);
    a.shadow[i] = shadow_ptrs.empty() ? nullptr : reinterpret_cast<void*>(shadow_ptrs[i]);
  }
  TORCH_CHECK(m.numel() == hi - lo && v.numel() == hi - lo, "ddp_zero_step: moment shards must have hi - lo elements");
  a.m = m.data_ptr<float>(), a.v = v.data_ptr<float>();
  a.lo = lo, a.hi = hi;
  a.h.kind = int(kind), a.h.first_step = first_step ? 1 : 0;
  a.h.lr = float(lr), a.h.beta1 = float(beta1), a.h.beta2 = float(beta2), a.h.eps = float(eps), a.h.decay = float(decay);
  a.h.clip = float(clip), a.h.step_size = float(step_size), a.h.inv_sqrt_bc2 = float(inv_sqrt_bc2);
  a.max_norm = float(max_norm), a.grad_mult = float(grad_mult);
  a.grads_mc = reinterpret_cast<const float*>(grads_mc);
  a.params_mc = reinterpret_cast<float*>(params_mc);
  a.shadow_mc = shadow_ptrs.empty() ? nullptr : reinterpret_cast<void*>(shadow_mc);
  pb::ddp_zero_step_launch(a, c, uint32_t(epoch), out_norm.has_value() ? out_norm->data_ptr<float>() : nullptr,
                           at::cuda::getCurrentDeviceProperties()->multiProcessorCount, at::cuda::getCurrentCUDAStream(device).stream());
  g_launches += 1;
}
void set_wsum(int64_t ctl_ptr, int device, double w, bool zero_sums) {
  c10::cuda::CUDAGuard guard(static_cast<c10::DeviceIndex>(device));
  pb::set_wsum(reinterpret_cast<uint32_t*>(ctl_ptr), float(w), zero_sums, at::cuda::getCurrentCUDAStream(device).stream());
  g_launches += 1;
}

long long launch_count() { return g_launches.load(); }
void reset_launch_count() { g_launches = 0; }
void add_launch_count(long long n) { g_launches += n; }  // launches replayed from a CUDA graph

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.doc() = "photon_b200 sm_100a kernels (tcgen05/TMEM/TMA GEMM + attention, fused norm/loss/optimizer, NVLink collectives)";
  m.def("gemm", &gemm, py::arg("a"), py::arg("b"), py::arg("d"), py::arg("a_mn") = 0, py::arg("b_mn") = 0, py::arg("epi") = 0,
        py::arg("bias") = py::none(), py::arg("aux") = py::none(), py::arg("d2") = py::none(), py::arg("accumulate") = false,
        py::arg("alpha") = 1.0, py::arg("cluster") = 0);
  m.def("gemm_fp8", &gemm_fp8, py::arg("a"), py::arg("b"), py::arg("d"), py::arg("a_mn"), py::arg("b_mn"), py::arg("epi"), py::arg("a_fmt"),
        py::arg("b_fmt"), py::arg("meta"), py::arg("role_a"), py::arg("role_b"), py::arg("bias") = py::none(), py::arg("aux") = py::none(),
        py::arg("d2") = py::none(), py::arg("accumulate") = false, py::arg("alpha") = 1.0, py::arg("cluster") = 0,
        py::arg("d8") = py::none(), py::arg("role_out") = -1);
  m.def("layernorm_fwd_q8", &layernorm_fwd_q8);
  m.def("mx_quantize", &mx_quantize, py::arg("x"), py::arg("rblk") = 0);
  m.def("gemm_mxfp8", &gemm_mxfp8, py::arg("a8"), py::arg("b8"), py::arg("d"), py::arg("sfa"), py::arg("sfb"), py::arg("bias") = py::none());
  m.def("colsum_quant", &colsum_quant, py::arg("dy"), py::arg("out_sum") = py::none(), py::arg("y8") = py::none(), py::arg("fmt") = 1,
        py::arg("meta") = py::none(), py::arg("role") = -1);
  m.def("fp8_quantize_segments", &fp8_quantize_segments);
  m.def("fp8_update_scales", &fp8_update_scales);
  m.def("attention_fwd", &attention_fwd, py::arg("qkv"), py::arg("out"), py::arg("lse"), py::arg("n_heads"), py::arg("scale"),
        py::arg("causal"), py::arg("alibi_slopes") = py::none());
  m.def("attention_bwd", &attention_bwd, py::arg("qkv"), py::arg("out"), py::arg("dout"), py::arg("lse"), py::arg("dqkv"), py::arg("delta"),
        py::arg("n_heads"), py::arg("scale"), py::arg("causal"), py::arg("alibi_slopes") = py::none());
  m.def("rope", &rope);
  m.def("embed_fwd", &embed_fwd);
  m.def("embed_bwd", &embed_bwd);
  m.def("layernorm_fwd", &layernorm_fwd);
  m.def("layernorm_bwd", &layernorm_bwd);
  m.def("col_sum", &col_sum);
  m.def("cross_entropy", &cross_entropy);
  m.def("flat_l2_norm", &flat_l2_norm);
  m.def("axpby", &axpby);
  m.def("cast_bf16", &cast_bf16);
  m.def("fused_optimizer", &fused_optimizer);
  m.def("embed_at", &embed_at);
  m.def("decode_attention_splits", &decode_attention_splits);
  m.def("decode_attention", &decode_attention, py::arg("q"), py::arg("kv"), py::arg("lengths"), py::arg("alibi_slopes"), py::arg("scale"),
        py::arg("n_heads"), py::arg("n_split"), py::arg("out"), py::arg("lse") = py::none());
  m.def("kv_write", &kv_write);
  m.def("argmax_rows", &argmax_rows);
  m.attr("DECODE_TILE_KEYS") = pb::DECODE_TILE_KEYS;
  m.def("ipc_alloc", &ipc_alloc);
  m.def("ipc_get_handle", &ipc_get_handle);
  m.def("ipc_open_handle", &ipc_open_handle);
  m.def("ipc_close", &ipc_close);
  m.def("ipc_free", &ipc_free);
  m.def("enable_peer_access", &enable_peer_access);
  m.def("tensor_from_ptr", &tensor_from_ptr);
  m.def("fed_round", &fed_round, py::arg("ctl_ptrs"), py::arg("rank"), py::arg("device"), py::arg("epoch"), py::arg("acc_ptrs"),
        py::arg("xg_ptrs"), py::arg("xs_ptrs"), py::arg("m_ptr"), py::arg("v_ptr"), py::arg("lo"), py::arg("hi"), py::arg("total"),
        py::arg("kind"), py::arg("avg_scale"), py::arg("lr"), py::arg("mu"), py::arg("eta"), py::arg("beta1"), py::arg("beta2"),
        py::arg("tau"), py::arg("round_t"), py::arg("sign_compat"), py::arg("acc_mc") = 0, py::arg("xg_mc") = 0,
        py::arg("seg_bounds") = py::none(), py::arg("seg_sums") = py::none(), py::arg("wsum") = -1.0, py::arg("zero_seg_sums") = false);
  m.def("set_comm_timeout_ms", [](long long ms) { g_comm_timeout_ms = ms < 0 ? 0 : ms; });
  m.def("comm_timeout_ms", []() { return g_comm_timeout_ms.load(); });
  m.def("ctl_status_word_offset", &pb::ctl_status_word_offset);
  m.def("ddp_allreduce", &ddp_allreduce, py::arg("ctl_ptrs"), py::arg("rank"), py::arg("device"), py::arg("epoch"), py::arg("buf_ptrs"),
        py::arg("lo"), py::arg("hi"), py::arg("out_norm") = py::none(), py::arg("buf_mc") = 0);
  m.def("zero3_reduce", &zero3_reduce, py::arg("ctl_ptrs"), py::arg("rank"), py::arg("device"), py::arg("epoch"), py::arg("stage_ptrs"),
        py::arg("stage_mc"), py::arg("dst"), py::arg("per"));
  m.def("memcpy_async", &memcpy_async);
  m.def("ddp_zero_step", &ddp_zero_step, py::arg("ctl_ptrs"), py::arg("rank"), py::arg("device"), py::arg("epoch"), py::arg("grad_ptrs"),
        py::arg("param_ptrs"), py::arg("shadow_ptrs"), py::arg("m"), py::arg("v"), py::arg("lo"), py::arg("hi"), py::arg("kind"),
        py::arg("first_step"), py::arg("lr"), py::arg("beta1"), py::arg("beta2"), py::arg("eps"), py::arg("decay"), py::arg("clip"),
        py::arg("step_size"), py::arg("inv_sqrt_bc2"), py::arg("max_norm"), py::arg("grad_mult"), py::arg("out_norm") = py::none(),
        py::arg("grads_mc") = 0, py::arg("params_mc") = 0, py::arg("shadow_mc") = 0);
  m.def("set_wsum", &set_wsum);
  m.def("ctl_sums_word_offset", &pb::ctl_sums_word_offset);
  m.def("launch_count", &launch_count);
  m.def("reset_launch_count", &reset_launch_count);
  m.def("add_launch_count", &add_launch_count);
  m.attr("CTL_WORDS") = pb::CTL_WORDS;
  m.attr("EPI_BF16") = int(pb::EPI_BF16);
  m.attr("EPI_RESIDUAL") = int(pb::EPI_RESIDUAL);
  m.attr("EPI_GELU_DUAL") = int(pb::EPI_GELU_DUAL);
  m.attr("EPI_DGELU") = int(pb::EPI_DGELU);
  m.attr("EPI_F32") = int(pb::EPI_F32);
  m.attr("EPI_GELU_GRAD") = int(pb::EPI_GELU_GRAD);
  m.attr("EPI_MUL") = int(pb::EPI_MUL);
  m.attr("EPI_GELU_GRAD_Q8") = int(pb::EPI_GELU_GRAD_Q8);
}
