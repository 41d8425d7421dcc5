// Memory-bound fused kernels of the MPT training step for sm_100a (everything that is not a GEMM or
// attention): embedding gather/scatter, LayerNorm fwd/bwd (+residual-gradient add), column reductions for
// bias / LN-affine gradients, fused cross-entropy (loss + in-place dlogits), flat-buffer L2 norm,
// ADOPT / DecoupledAdamW multi-tensor step with bf16 shadow emit, axpby for the streaming client mean.
// All are 128-bit vectorised, one pass over HBM; they replace the ATen kernel sequences the reference
// reaches through torch (SURVEY §2.5 K1, K2, K9, K11, K12, K14).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <cstdlib>
#include <stdexcept>
#include <string>

#include "fused_ops.h"
#include "optim_dev.cuh"
#include "ptx.cuh"

namespace pb {

namespace {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffff, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffff, v, o));
  return v;
}
__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y), c = unpack_bf16(u.z), d = unpack_bf16(u.w);
  f[0] = a.x, f[1] = a.y, f[2] = b.x, f[3] = b.y, f[4] = c.x, f[5] = c.y, f[6] = d.x, f[7] = d.y;
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint4 u;
  u.x = pack_bf16(f[0], f[1]), u.y = pack_bf16(f[2], f[3]), u.z = pack_bf16(f[4], f[5]), u.w = pack_bf16(f[6], f[7]);
  return u;
}

// ------------------------------------------------------------------ embedding
// h[t,:] = wte[ids[t],:] + wpe[t % S,:]      (bf16 tables = compute shadow of the fp32 masters)
// With `pos` (int32 [T], decoding: one row per sequence at its own position) the position is pos[t], clamped to [0, S).
__global__ void embed_fwd_kernel(const int64_t* __restrict__ ids, const __nv_bfloat16* __restrict__ wte,
                                 const __nv_bfloat16* __restrict__ wpe, __nv_bfloat16* __restrict__ out, long long T,
                                 int S, int d, int V, const int* __restrict__ pos) {
  const int vec = d / 8;
  for (long long t = blockIdx.x; t < T; t += gridDim.x) {
    long long id = ids[t];
    id = id < 0 ? 0 : (id >= V ? V - 1 : id);
    const uint4* a = reinterpret_cast<const uint4*>(wte + id * d);
    const int p = pos ? min(max(pos[t], 0), S - 1) : int(t % S);
    const uint4* b = wpe ? reinterpret_cast<const uint4*>(wpe + (long long)p * d) : nullptr;
    uint4* o = reinterpret_cast<uint4*>(out + t * d);
    for (int i = threadIdx.x; i < vec; i += blockDim.x) {
      float x[8], y[8];
      unpack8(__ldg(a + i), x);
      if (b) {
        unpack8(__ldg(b + i), y);
#pragma unroll
        for (int k = 0; k < 8; ++k) x[k] += y[k];
      }
      o[i] = pack8(x);
    }
  }
}

// dwte[ids[t],:] += dh[t,:]  (vector RED), one block per token
__global__ void embed_bwd_wte_kernel(const int64_t* __restrict__ ids, const __nv_bfloat16* __restrict__ dh,
                                     float* __restrict__ dwte, long long T, int d, int V) {
  const int vec = d / 8;
  for (long long t = blockIdx.x; t < T; t += gridDim.x) {
    long long id = ids[t];
    if (id < 0 || id >= V) continue;
    const uint4* g = reinterpret_cast<const uint4*>(dh + t * d);
    float* dst = dwte + id * d;
    for (int i = threadIdx.x; i < vec; i += blockDim.x) {
      float x[8];
      unpack8(g[i], x);
      float* p = dst + i * 8;
      asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(x[0]), "f"(x[1]), "f"(x[2]), "f"(x[3])
                   : "memory");
      asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p + 4), "f"(x[4]), "f"(x[5]), "f"(x[6]),
                   "f"(x[7])
                   : "memory");
    }
  }
}
// dwpe[s,:] += sum_b dh[b*S+s,:]   (no atomics: one block owns one position)
__global__ void embed_bwd_wpe_kernel(const __nv_bfloat16* __restrict__ dh, float* __restrict__ dwpe, int Bsz, int S,
                                     int d) {
  const int s = blockIdx.x;
  const int vec = d / 8;
  for (int i = threadIdx.x; i < vec; i += blockDim.x) {
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int b = 0; b < Bsz; ++b) {
      float x[8];
      unpack8(reinterpret_cast<const uint4*>(dh + ((long long)b * S + s) * d)[i], x);
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[k] += x[k];
    }
    float4* o = reinterpret_cast<float4*>(dwpe + (long long)s * d + i * 8);
    float4 o0 = o[0], o1 = o[1];
    o0.x += acc[0], o0.y += acc[1], o0.z += acc[2], o0.w += acc[3];
    o1.x += acc[4], o1.y += acc[5], o1.z += acc[6], o1.w += acc[7];
    o[0] = o0, o[1] = o1;
  }
}

// ------------------------------------------------------------------ LayerNorm (one warp per row, row in registers)
constexpr int LN_MAXCH = 16;  // 16 chunks x 32 lanes x 8 elems = d <= 4096

template <int LN_NCH>
__global__ void __launch_bounds__(256) ln_fwd_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ gamma,
                                                      const float* __restrict__ beta, __nv_bfloat16* __restrict__ y,
                                                      float* __restrict__ mean, float* __restrict__ rstd, long long T,
                                                      int d, float eps) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= T) return;
  const uint4* xr = reinterpret_cast<const uint4*>(x + row * d);
  uint4 buf[LN_NCH];
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < LN_NCH; ++c) {
    const int e = c * 256 + lane * 8;
    if (e < d) {
      buf[c] = xr[c * 32 + lane];
      float f[8];
      unpack8(buf[c], f);
#pragma unroll
      for (int k = 0; k < 8; ++k) s += f[k];
    }
  }
  const float mu = warp_sum(s) / d;
  float ss = 0.f;
#pragma unroll
  for (int c = 0; c < LN_NCH; ++c) {
    const int e = c * 256 + lane * 8;
    if (e < d) {
      float f[8];
      unpack8(buf[c], f);
#pragma unroll
      for (int k = 0; k < 8; ++k) ss += (f[k] - mu) * (f[k] - mu);
    }
  }
  const float rs = rsqrtf(warp_sum(ss) / d + eps);
  if (lane == 0) {
    mean[row] = mu;
    rstd[row] = rs;
  }
  uint4* yr = reinterpret_cast<uint4*>(y + row * d);
#pragma unroll
  for (int c = 0; c < LN_NCH; ++c) {
    const int e = c * 256 + lane * 8;
    if (e < d) {
      float f[8];
      unpack8(buf[c], f);
      const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma + e)), g1 = __ldg(reinterpret_cast<const float4*>(gamma + e + 4));
      float4 b0 = make_float4(0, 0, 0, 0), b1 = b0;
      if (beta) b0 = __ldg(reinterpret_cast<const float4*>(beta + e)), b1 = __ldg(reinterpret_cast<const float4*>(beta + e + 4));
      const float g[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
      const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int k = 0; k < 8; ++k) f[k] = (f[k] - mu) * rs * g[k] + b[k];
      yr[c * 32 + lane] = pack8(f);
    }
  }
}

// dx = rstd * (dy*g - mean(dy*g) - xhat * mean(dy*g*xhat))  [+ dres]   (row-wise part of LN backward)
template <int LN_NCH>
__global__ void __launch_bounds__(256) ln_bwd_dx_kernel(const __nv_bfloat16* __restrict__ dy, const __nv_bfloat16* __restrict__ x,
                                                         const float* __restrict__ gamma, const float* __restrict__ mean,
                                                         const float* __restrict__ rstd, const __nv_bfloat16* __restrict__ dres,
                                                         __nv_bfloat16* __restrict__ dx, long long T, int d) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= T) return;
  const uint4* xr = reinterpret_cast<const uint4*>(x + row * d);
  const uint4* gr = reinterpret_cast<const uint4*>(dy + row * d);
  const float mu = mean[row], rs = rstd[row];
  uint4 bx[LN_NCH], bg[LN_NCH];
  float c1 = 0.f, c2 = 0.f;
#pragma unroll
  for (int c = 0; c < LN_NCH; ++c) {
    const int e = c * 256 + lane * 8;
    if (e < d) {
      bx[c] = xr[c * 32 + lane];
      bg[c] = gr[c * 32 + lane];
      float fx[8], fg[8];
      unpack8(bx[c], fx);
      unpack8(bg[c], fg);
      const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma + e)), g1 = __ldg(reinterpret_cast<const float4*>(gamma + e + 4));
      const float g[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float dxh = fg[k] * g[k];
        c1 += dxh;
        c2 += dxh * (fx[k] - mu) * rs;
      }
    }
  }
  c1 = warp_sum(c1) / d;
  c2 = warp_sum(c2) / d;
  uint4* outr = reinterpret_cast<uint4*>(dx + row * d);
  const uint4* rr = dres ? reinterpret_cast<const uint4*>(dres + row * d) : nullptr;
#pragma unroll
  for (int c = 0; c < LN_NCH; ++c) {
    const int e = c * 256 + lane * 8;
    if (e < d) {
      float fx[8], fg[8], fr[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      unpack8(bx[c], fx);
      unpack8(bg[c], fg);
      if (rr) unpack8(rr[c * 32 + lane], fr);
      const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma + e)), g1 = __ldg(reinterpret_cast<const float4*>(gamma + e + 4));
      const float g[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float xh = (fx[k] - mu) * rs;
        fx[k] = rs * (fg[k] * g[k] - c1 - xh * c2) + fr[k];
      }
      outr[c * 32 + lane] = pack8(fx);
    }
  }
}

// Same row-wise dx, plus the column reductions dbeta[j] += sum_t dy[t,j], dgamma[j] += sum_t dy[t,j] * xhat[t,j] in the SAME
// pass (persistent warps keep per-lane column partials in registers; one smem reduction + one atomicAdd per column per
// block at the end). Saves the second read of dy and x that a separate column-reduce kernel needs. d <= 1024.
template <int LN_NCH>
__global__ void __launch_bounds__(256, 2) ln_bwd_fused_kernel(const __nv_bfloat16* __restrict__ dy, const __nv_bfloat16* __restrict__ x,
                                                            const float* __restrict__ gamma, const float* __restrict__ mean,
                                                            const float* __restrict__ rstd, const __nv_bfloat16* __restrict__ dres,
                                                            __nv_bfloat16* __restrict__ dx, float* __restrict__ dgamma,
                                                            float* __restrict__ dbeta, long long T, int d) {
  __shared__ float sred[8][LN_NCH * 256];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const long long nwarps = (long long)gridDim.x * 8;
  float ag[LN_NCH][8], ab[LN_NCH][8];
#pragma unroll
  for (int c = 0; c < LN_NCH; ++c)
#pragma unroll
    for (int k = 0; k < 8; ++k) ag[c][k] = 0.f, ab[c][k] = 0.f;
  auto load_gamma = [&](int c, float (&g)[8]) {   // L1-resident after the first row; keeping it in registers costs occupancy
    const int e = c * 256 + lane * 8;
    if (e < d) {
      const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma + e)), g1 = __ldg(reinterpret_cast<const float4*>(gamma + e + 4));
      g[0] = g0.x, g[1] = g0.y, g[2] = g0.z, g[3] = g0.w, g[4] = g1.x, g[5] = g1.y, g[6] = g1.z, g[7] = g1.w;
    } else {
#pragma unroll
      for (int k = 0; k < 8; ++k) g[k] = 0.f;
    }
  };
  for (long long row = (long long)blockIdx.x * 8 + w; row < T; row += nwarps) {
    const uint4* xr = reinterpret_cast<const uint4*>(x + row * d);
    const uint4* gr = reinterpret_cast<const uint4*>(dy + row * d);
    const float mu = mean[row], rs = rstd[row];
    uint4 bx[LN_NCH], bg[LN_NCH];
    float c1 = 0.f, c2 = 0.f;
#pragma unroll
    for (int c = 0; c < LN_NCH; ++c) {
      const int e = c * 256 + lane * 8;
      if (e < d) {
        bx[c] = xr[c * 32 + lane];
        bg[c] = gr[c * 32 + lane];
      } else {
        bx[c] = make_uint4(0, 0, 0, 0), bg[c] = make_uint4(0, 0, 0, 0);
      }
    }
#pragma unroll
    for (int c = 0; c < LN_NCH; ++c) {
      float fx[8], fg[8], g[8];
      unpack8(bx[c], fx);
      unpack8(bg[c], fg);
      load_gamma(c, g);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float xh = (fx[k] - mu) * rs;
        const float dxh = fg[k] * g[k];
        c1 += dxh;
        c2 += dxh * xh;
        ab[c][k] += fg[k];
        ag[c][k] += fg[k] * xh;
      }
    }
    c1 = warp_sum(c1) / d;
    c2 = warp_sum(c2) / d;
    uint4* outr = reinterpret_cast<uint4*>(dx + row * d);
    const uint4* rr = dres ? reinterpret_cast<const uint4*>(dres + row * d) : nullptr;
#pragma unroll
    for (int c = 0; c < LN_NCH; ++c) {
      const int e = c * 256 + lane * 8;
      if (e < d) {
        float fx[8], fg[8], g[8], fr[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        unpack8(bx[c], fx);
        unpack8(bg[c], fg);
        load_gamma(c, g);
        if (rr) unpack8(rr[c * 32 + lane], fr);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const float xh = (fx[k] - mu) * rs;
          fx[k] = rs * (fg[k] * g[k] - c1 - xh * c2) + fr[k];
        }
        outr[c * 32 + lane] = pack8(fx);
      }
    }
  }
  // block reduction of the column partials: dbeta then dgamma through the same smem
#pragma unroll
  for (int pass = 0; pass < 2; ++pass) {
    __syncthreads();
#pragma unroll
    for (int c = 0; c < LN_NCH; ++c)
#pragma unroll
      for (int k = 0; k < 8; ++k) sred[w][c * 256 + lane * 8 + k] = pass == 0 ? ab[c][k] : ag[c][k];
    __syncthreads();
    float* out = pass == 0 ? dbeta : dgamma;
    if (out) {
      for (int j = threadIdx.x; j < d; j += 256) {
        float t = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) t += sred[i][j];
        atomicAdd(out + j, t);
      }
    }
  }
}

// Column reductions over rows: out_sum[j] += sum_t dy[t,j];  (optional) out_dot[j] += sum_t dy[t,j]*xhat[t,j].
// Used for bias gradients (x == nullptr) and for LN dgamma/dbeta. Block = 8 warps x 256 columns.
__global__ void __launch_bounds__(256) col_reduce_kernel(const __nv_bfloat16* __restrict__ dy, long long ld,
                                                          const __nv_bfloat16* __restrict__ x, const float* __restrict__ mean,
                                                          const float* __restrict__ rstd, float* __restrict__ out_sum,
                                                          float* __restrict__ out_dot, long long T, int d, int rows_per_block) {
  __shared__ float ssum[8][256];
  __shared__ float sdot[8][256];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int col = blockIdx.x * 256 + lane * 8;
  const long long r0 = (long long)blockIdx.y * rows_per_block;
  const long long r1 = r0 + rows_per_block < T ? r0 + rows_per_block : T;
  float as[8] = {0, 0, 0, 0, 0, 0, 0, 0}, ad[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (col < d) {
    // 4 independent 16-byte loads per thread in flight (the row loop alone keeps one: ~16 KiB per SM, a quarter of what
    // HBM3e needs to stay busy)
    long long r = r0 + w;
    for (; r + 24 < r1; r += 32) {
      uint4 q[4], qx[4];
      float mu[4], rs[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        q[u] = *reinterpret_cast<const uint4*>(dy + (r + 8 * u) * ld + col);
        if (x) {
          qx[u] = *reinterpret_cast<const uint4*>(x + (r + 8 * u) * (long long)d + col);
          mu[u] = mean[r + 8 * u], rs[u] = rstd[r + 8 * u];
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float g[8];
        unpack8(q[u], g);
        if (x) {
          float fx[8];
          unpack8(qx[u], fx);
#pragma unroll
          for (int k = 0; k < 8; ++k) ad[k] += g[k] * (fx[k] - mu[u]) * rs[u];
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) as[k] += g[k];
      }
    }
    for (; r < r1; r += 8) {
      float g[8];
      unpack8(*reinterpret_cast<const uint4*>(dy + r * ld + col), g);
      if (x) {
        float fx[8];
        unpack8(*reinterpret_cast<const uint4*>(x + r * (long long)d + col), fx);
        const float mu = mean[r], rs = rstd[r];
#pragma unroll
        for (int k = 0; k < 8; ++k) ad[k] += g[k] * (fx[k] - mu) * rs;
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) as[k] += g[k];
    }
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    ssum[w][lane * 8 + k] = as[k];
    sdot[w][lane * 8 + k] = ad[k];
  }
  __syncthreads();
  const int c = threadIdx.x;
  if (blockIdx.x * 256 + c < d) {
    float s = 0.f, t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += ssum[i][c], t += sdot[i][c];
    atomicAdd(out_sum + blockIdx.x * 256 + c, s);
    if (out_dot) atomicAdd(out_dot + blockIdx.x * 256 + c, t);
  }
}

// ------------------------------------------------------------------ fused cross-entropy
// One block per row of logits[Tc, V] (bf16). Pass 1: online max / sum-exp (+argmax). Pass 2 (training):
// overwrite the row with dlogits = (softmax - onehot) * grad_scale (zero for ignored rows).
// stats[0] += sum loss, stats[1] += #valid, stats[2] += #correct, stats[3] += sum unigram loss  (fp64)
__global__ void __launch_bounds__(256) ce_kernel(__nv_bfloat16* __restrict__ logits, long long ld, const int64_t* __restrict__ targets,
                                                  int V, float grad_scale, int write_grad, double* __restrict__ stats,
                                                  float* __restrict__ row_lse, const float* __restrict__ unigram_logp) {
  __shared__ float sm[8], ss[8];
  __shared__ int si[8];
  __shared__ float bm, bs;
  __shared__ int bi;
  const long long row = blockIdx.x;
  __nv_bfloat16* lr = logits + row * ld;
  const long long tgt = targets[row];
  const bool valid = tgt >= 0 && tgt < V;
  const int vec = V / 8;
  float m = -INFINITY, s = 0.f;
  int am = 0;
  for (int i = threadIdx.x; i < vec; i += blockDim.x) {
    float f[8];
    unpack8(reinterpret_cast<const uint4*>(lr)[i], f);
    float cm = f[0];
    int ci = 0;
#pragma unroll
    for (int k = 1; k < 8; ++k)
      if (f[k] > cm) cm = f[k], ci = k;
    if (cm > m) {
      s *= __expf(m - cm);
      m = cm;
      am = i * 8 + ci;
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) s += __expf(f[k] - m);
  }
  // warp + block combine of (m, s, argmax)
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffff, m, o), os = __shfl_xor_sync(0xffffffff, s, o);
    const int oi = __shfl_xor_sync(0xffffffff, am, o);
    const float nm = fmaxf(m, om);
    s = (m == -INFINITY ? 0.f : s * __expf(m - nm)) + (om == -INFINITY ? 0.f : os * __expf(om - nm));
    if (om > m || (om == m && oi < am)) am = oi;
    m = nm;
  }
  if (lane == 0) sm[w] = m, ss[w] = s, si[w] = am;
  __syncthreads();
  if (threadIdx.x == 0) {
    float M = sm[0], S = ss[0];
    int I = si[0];
    for (int i = 1; i < 8; ++i) {
      const float nm = fmaxf(M, sm[i]);
      S = (M == -INFINITY ? 0.f : S * __expf(M - nm)) + (sm[i] == -INFINITY ? 0.f : ss[i] * __expf(sm[i] - nm));
      if (sm[i] > M || (sm[i] == M && si[i] < I)) I = si[i];
      M = nm;
    }
    bm = M, bs = S, bi = I;
    const float lse = M + __logf(S);
    if (row_lse) row_lse[row] = lse;
    if (valid) {
      const float lt = __bfloat162float(lr[tgt]);
      atomicAdd(stats + 0, double(lse - lt));
      atomicAdd(stats + 1, 1.0);
      if (I == tgt) atomicAdd(stats + 2, 1.0);
      if (unigram_logp) atomicAdd(stats + 3, double(-unigram_logp[tgt]));
    }
  }
  __syncthreads();
  if (!write_grad) return;
  const float M = bm, inv = grad_scale / bs;
  for (int i = threadIdx.x; i < vec; i += blockDim.x) {
    float f[8];
    uint4* p = reinterpret_cast<uint4*>(lr) + i;
    unpack8(*p, f);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float g = valid ? __expf(f[k] - M) * inv : 0.f;
      if (valid && i * 8 + k == tgt) g -= grad_scale;
      f[k] = g;
    }
    *p = pack8(f);
  }
}

// Same contract, ONE read of the logits: the whole row (V bf16 = 100 KB for the GPT-NeoX vocabulary) is pulled into shared
// memory by bulk async copies (cp.async.bulk on an mbarrier), both passes run out of shared memory and only the gradient goes back
// to HBM — 2 instead of 3 row transfers per row. Two CTAs fit on an SM, so one row's copy overlaps the other's arithmetic.
__global__ void __launch_bounds__(512) ce_smem_kernel(__nv_bfloat16* __restrict__ logits, long long ld, const int64_t* __restrict__ targets,
                                                       int V, float grad_scale, int write_grad, double* __restrict__ stats,
                                                       float* __restrict__ row_lse, const float* __restrict__ unigram_logp) {
  extern __shared__ __align__(128) uint8_t ce_smem[];
  uint4* srow = reinterpret_cast<uint4*>(ce_smem);
  __shared__ uint64_t bar;
  __shared__ float sm[16], ss[16];
  __shared__ int si[16];
  __shared__ float bm, bs;
  const long long row = blockIdx.x;
  __nv_bfloat16* lr = logits + row * ld;
  const long long tgt = targets[row];
  const bool valid = tgt >= 0 && tgt < V;
  const int vec = V / 8;
  const uint32_t bytes = uint32_t(V) * 2u;
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    fence_barrier_init();
    mbar_expect_tx(&bar, bytes);
    for (uint32_t off = 0; off < bytes; off += 32768u) {   // bulk copies of <= 32 KiB, all counted on the one barrier
      const uint32_t n = bytes - off < 32768u ? bytes - off : 32768u;
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(ce_smem + off)),
                   "l"(reinterpret_cast<uint64_t>(reinterpret_cast<const uint8_t*>(lr) + off)), "r"(n), "r"(smem_u32(&bar))
                   : "memory");
    }
  }
  __syncthreads();
  mbar_wait(&bar, 0);
  float m = -INFINITY, s = 0.f;
  int am = 0;
  for (int i = threadIdx.x; i < vec; i += blockDim.x) {
    float f[8];
    unpack8(srow[i], f);
    float cm = f[0];
    int ci = 0;
#pragma unroll
    for (int k = 1; k < 8; ++k)
      if (f[k] > cm) cm = f[k], ci = k;
    if (cm > m) {
      s *= __expf(m - cm);
      m = cm;
      am = i * 8 + ci;
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) s += __expf(f[k] - m);
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffff, m, o), os = __shfl_xor_sync(0xffffffff, s, o);
    const int oi = __shfl_xor_sync(0xffffffff, am, o);
    const float nm = fmaxf(m, om);
    s = (m == -INFINITY ? 0.f : s * __expf(m - nm)) + (om == -INFINITY ? 0.f : os * __expf(om - nm));
    if (om > m || (om == m && oi < am)) am = oi;
    m = nm;
  }
  if (lane == 0) sm[w] = m, ss[w] = s, si[w] = am;
  __syncthreads();
  if (threadIdx.x == 0) {
    float M = sm[0], S = ss[0];
    int I = si[0];
    for (int i = 1; i < nw; ++i) {
      const float nm = fmaxf(M, sm[i]);
      S = (M == -INFINITY ? 0.f : S * __expf(M - nm)) + (sm[i] == -INFINITY ? 0.f : ss[i] * __expf(sm[i] - nm));
      if (sm[i] > M || (sm[i] == M && si[i] < I)) I = si[i];
      M = nm;
    }
    bm = M, bs = S;
    const float lse = M + __logf(S);
    if (row_lse) row_lse[row] = lse;
    if (valid) {
      const float lt = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(ce_smem)[tgt]);
      atomicAdd(stats + 0, double(lse - lt));
      atomicAdd(stats + 1, 1.0);
      if (I == tgt) atomicAdd(stats + 2, 1.0);
      if (unigram_logp) atomicAdd(stats + 3, double(-unigram_logp[tgt]));
    }
  }
  __syncthreads();
  if (!write_grad) return;
  const float M = bm, inv = grad_scale / bs;
  for (int i = threadIdx.x; i < vec; i += blockDim.x) {
    float f[8];
    unpack8(srow[i], f);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float g = valid ? __expf(f[k] - M) * inv : 0.f;
      if (valid && i * 8 + k == tgt) g -= grad_scale;
      f[k] = g;
    }
    reinterpret_cast<uint4*>(lr)[i] = pack8(f);
  }
}

// ------------------------------------------------------------------ flat helpers
__global__ void sqnorm_kernel(const float* __restrict__ x, long long n, double* __restrict__ out) {
  __shared__ float sh[32];
  float acc = 0.f;
  const long long n4 = n / 4;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(x)[i];
    acc += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? sh[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) atomicAdd(out, double(v));
  }
}
__global__ void sqrt_finalize_kernel(const double* __restrict__ in, float* __restrict__ out) { *out = float(sqrt(*in)); }

__global__ void axpby_kernel(float* __restrict__ acc, const float* __restrict__ x, float a, float b, long long n4) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 u = reinterpret_cast<float4*>(acc)[i];
    const float4 v = reinterpret_cast<const float4*>(x)[i];
    u.x = a * u.x + b * v.x, u.y = a * u.y + b * v.y, u.z = a * u.z + b * v.z, u.w = a * u.w + b * v.w;
    reinterpret_cast<float4*>(acc)[i] = u;
  }
}
__global__ void cast_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, long long n4) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(src)[i];
    uint2 o;
    o.x = pack_bf16(v.x, v.y), o.y = pack_bf16(v.z, v.w);
    reinterpret_cast<uint2*>(dst)[i] = o;
  }
}

// ------------------------------------------------------------------ fused optimizers (flat fp32 planes)
// kind 0 = ADOPT, 1 = DecoupledAdamW, 2 = SGD. grad_mult (device scalar, may be null) multiplies every
// gradient (clip coefficient x 1/loss-scale) so clipping needs no host round trip.
__global__ void __launch_bounds__(256) optim_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                     float* __restrict__ v, __nv_bfloat16* __restrict__ shadow, long long n4,
                                                     OptimHyper h, const float* __restrict__ grad_mult) {
  const float gm = grad_mult ? *grad_mult : 1.0f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 P = reinterpret_cast<float4*>(p)[i];
    float4 G = reinterpret_cast<const float4*>(g)[i];
    float pp[4] = {P.x, P.y, P.z, P.w};
    const float gg[4] = {G.x * gm, G.y * gm, G.z * gm, G.w * gm};
    float mm[4] = {0.f, 0.f, 0.f, 0.f}, vv[4] = {0.f, 0.f, 0.f, 0.f};
    if (h.kind != 2) {
      const float4 Mv = reinterpret_cast<float4*>(m)[i];
      const float4 Vv = reinterpret_cast<float4*>(v)[i];
      mm[0] = Mv.x, mm[1] = Mv.y, mm[2] = Mv.z, mm[3] = Mv.w;
      vv[0] = Vv.x, vv[1] = Vv.y, vv[2] = Vv.z, vv[3] = Vv.w;
    }
    optim_update4(pp, gg, mm, vv, h);
    if (h.kind != 2) {
      reinterpret_cast<float4*>(m)[i] = make_float4(mm[0], mm[1], mm[2], mm[3]);
      reinterpret_cast<float4*>(v)[i] = make_float4(vv[0], vv[1], vv[2], vv[3]);
    }
    reinterpret_cast<float4*>(p)[i] = make_float4(pp[0], pp[1], pp[2], pp[3]);
    if (shadow) {
      uint2 o;
      o.x = pack_bf16(pp[0], pp[1]), o.y = pack_bf16(pp[2], pp[3]);
      reinterpret_cast<uint2*>(shadow)[i] = o;
    }
  }
}

inline int grid_for(long long work_items, int block, int max_blocks = 148 * 8) {
  long long b = (work_items + block - 1) / block;
  if (b < 1) b = 1;
  return int(b < max_blocks ? b : max_blocks);
}

}  // namespace

#define PB_CHECK_LAUNCH(name)                                                                          \
  do {                                                                                                 \
    cudaError_t e__ = cudaGetLastError();                                                              \
    if (e__ != cudaSuccess) throw std::runtime_error(std::string(name " launch: ") + cudaGetErrorString(e__)); \
  } while (0)

void embed_fwd(const int64_t* ids, const void* wte, const void* wpe, void* out, long long T, int S, int d, int V, cudaStream_t st,
               const int* pos) {
  embed_fwd_kernel<<<grid_for(T, 1, 148 * 16), 128, 0, st>>>(ids, (const __nv_bfloat16*)wte, (const __nv_bfloat16*)wpe,
                                                            (__nv_bfloat16*)out, T, S, d, V, pos);
  PB_CHECK_LAUNCH("embed_fwd");
}
void embed_bwd(const int64_t* ids, const void* dh, float* dwte, float* dwpe, long long T, int S, int d, int V, cudaStream_t st) {
  embed_bwd_wte_kernel<<<grid_for(T, 1, 148 * 16), 128, 0, st>>>(ids, (const __nv_bfloat16*)dh, dwte, T, d, V);
  PB_CHECK_LAUNCH("embed_bwd_wte");
  if (dwpe) {
    embed_bwd_wpe_kernel<<<S, 128, 0, st>>>((const __nv_bfloat16*)dh, dwpe, int(T / S), S, d);
    PB_CHECK_LAUNCH("embed_bwd_wpe");
  }
}
void layernorm_fwd(const void* x, const float* gamma, const float* beta, void* y, float* mean, float* rstd, long long T, int d,
                   float eps, cudaStream_t st) {
  if (d % 8 || d > LN_MAXCH * 256) throw std::runtime_error("layernorm: d must be a multiple of 8 and <= 4096");
  const int nch = (d + 255) / 256;
#define PB_LN_FWD(N)                                                                                                            \
  if (nch <= N) {                                                                                                               \
    ln_fwd_kernel<N><<<int((T + 7) / 8), 256, 0, st>>>((const __nv_bfloat16*)x, gamma, beta, (__nv_bfloat16*)y, mean, rstd, T, d, eps); \
    PB_CHECK_LAUNCH("layernorm_fwd");                                                                                           \
    return;                                                                                                                     \
  }
  PB_LN_FWD(1) PB_LN_FWD(2) PB_LN_FWD(3) PB_LN_FWD(4) PB_LN_FWD(6) PB_LN_FWD(8) PB_LN_FWD(10) PB_LN_FWD(12) PB_LN_FWD(16)
#undef PB_LN_FWD
}
void col_reduce(const void* dy, long long ld, const void* x, const float* mean, const float* rstd, float* out_sum, float* out_dot,
                long long T, int d, cudaStream_t st) {
  const int col_blocks = (d + 255) / 256;
  int strips = (148 * 4 + col_blocks - 1) / col_blocks;
  if (strips > T) strips = int(T);
  const int rows_per = int((T + strips - 1) / strips);
  dim3 grid(col_blocks, int((T + rows_per - 1) / rows_per));
  col_reduce_kernel<<<grid, 256, 0, st>>>((const __nv_bfloat16*)dy, ld, (const __nv_bfloat16*)x, mean, rstd, out_sum, out_dot, T, d,
                                          rows_per);
  PB_CHECK_LAUNCH("col_reduce");
}
void layernorm_bwd(const void* dy, const void* x, const float* gamma, const float* mean, const float* rstd, const void* dres, void* dx,
                   float* dgamma, float* dbeta, long long T, int d, cudaStream_t st) {
  if (d % 8 || d > LN_MAXCH * 256) throw std::runtime_error("layernorm: d must be a multiple of 8 and <= 4096");
  const int nch = (d + 255) / 256;
  if ((dgamma || dbeta) && nch <= 4) {
    // d <= 1024: dx and the dgamma / dbeta column sums in ONE pass over dy and x
    const int grid = int(std::min<long long>((T + 7) / 8, 148 * 2));   // 2 resident blocks per SM
#define PB_LN_FUSED(N)                                                                                                      \
  if (nch <= N) {                                                                                                           \
    ln_bwd_fused_kernel<N><<<grid, 256, 0, st>>>((const __nv_bfloat16*)dy, (const __nv_bfloat16*)x, gamma, mean, rstd,           \
                                                 (const __nv_bfloat16*)dres, (__nv_bfloat16*)dx, dgamma, dbeta, T, d);      \
    PB_CHECK_LAUNCH("layernorm_bwd_fused");                                                                                 \
    return;                                                                                                                 \
  }
    PB_LN_FUSED(1) PB_LN_FUSED(2) PB_LN_FUSED(3) PB_LN_FUSED(4)
#undef PB_LN_FUSED
  }
  bool done = false;
#define PB_LN_BWD(N)                                                                                                  \
  if (!done && nch <= N) {                                                                                            \
    ln_bwd_dx_kernel<N><<<int((T + 7) / 8), 256, 0, st>>>((const __nv_bfloat16*)dy, (const __nv_bfloat16*)x, gamma, mean, rstd, \
                                                          (const __nv_bfloat16*)dres, (__nv_bfloat16*)dx, T, d);      \
    done = true;                                                                                                      \
  }
  PB_LN_BWD(1) PB_LN_BWD(2) PB_LN_BWD(3) PB_LN_BWD(4) PB_LN_BWD(6) PB_LN_BWD(8) PB_LN_BWD(10) PB_LN_BWD(12) PB_LN_BWD(16)
#undef PB_LN_BWD
  PB_CHECK_LAUNCH("layernorm_bwd_dx");
  if (dgamma || dbeta) col_reduce(dy, d, x, mean, rstd, dbeta, dgamma, T, d, st);
}
void cross_entropy(void* logits, long long ld, const int64_t* targets, long long rows, int V, float grad_scale, bool write_grad,
                   double* stats, float* row_lse, const float* unigram_logp, cudaStream_t st) {
  if (V % 8) throw std::runtime_error("cross_entropy: V must be a multiple of 8");
  const size_t row_bytes = size_t(V) * 2;
  static const bool smem_path = [] { const char* e = std::getenv("PB_CE_SMEM"); return !(e && e[0] == '0'); }();
  if (smem_path && row_bytes <= 200 * 1024 && (ld * 2) % 16 == 0 && (reinterpret_cast<uintptr_t>(logits) & 15) == 0) {
    // the row lives in shared memory between the two passes: one HBM read of the logits instead of two
    static bool configured = false;
    if (!configured) {
      cudaError_t e = cudaFuncSetAttribute(ce_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      if (e != cudaSuccess) throw std::runtime_error(std::string("cross_entropy smem attr: ") + cudaGetErrorString(e));
      configured = true;
    }
    ce_smem_kernel<<<int(rows), 512, row_bytes, st>>>((__nv_bfloat16*)logits, ld, targets, V, grad_scale, write_grad ? 1 : 0, stats, row_lse,
                                                      unigram_logp);
    PB_CHECK_LAUNCH("cross_entropy");
    return;
  }
  ce_kernel<<<int(rows), 256, 0, st>>>((__nv_bfloat16*)logits, ld, targets, V, grad_scale, write_grad ? 1 : 0, stats, row_lse,
                                       unigram_logp);
  PB_CHECK_LAUNCH("cross_entropy");
}
void flat_sqnorm(const float* x, long long n, double* out_accum, cudaStream_t st) {
  sqnorm_kernel<<<grid_for(n / 4, 256, 148 * 4), 256, 0, st>>>(x, n, out_accum);
  PB_CHECK_LAUNCH("flat_sqnorm");
}
void sqrt_finalize(const double* in, float* out, cudaStream_t st) {
  sqrt_finalize_kernel<<<1, 1, 0, st>>>(in, out);
  PB_CHECK_LAUNCH("sqrt_finalize");
}
void axpby(float* acc, const float* x, float a, float b, long long n, cudaStream_t st) {
  axpby_kernel<<<grid_for(n / 4, 256, 148 * 8), 256, 0, st>>>(acc, x, a, b, n / 4);
  PB_CHECK_LAUNCH("axpby");
}
void cast_fp32_to_bf16(const float* src, void* dst, long long n, cudaStream_t st) {
  cast_bf16_kernel<<<grid_for(n / 4, 256, 148 * 8), 256, 0, st>>>(src, (__nv_bfloat16*)dst, n / 4);
  PB_CHECK_LAUNCH("cast_bf16");
}
void fused_optimizer(float* p, const float* g, float* m, float* v, void* shadow, long long n, const OptimHyper& h,
                     const float* grad_mult, cudaStream_t st) {
  optim_kernel<<<grid_for(n / 4, 256, 148 * 8), 256, 0, st>>>(p, g, m, v, (__nv_bfloat16*)shadow, n / 4, h, grad_mult);
  PB_CHECK_LAUNCH("fused_optimizer");
}

}  // namespace pb
