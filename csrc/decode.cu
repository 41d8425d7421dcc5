// Kernels of KV-cached greedy decoding for sm_100a: split-KV decode attention over a ragged cache ("flash-decoding"),
// the KV-cache write fused with RoPE at explicit positions, and the row argmax over the vocabulary. All take bf16 and
// compute in fp32. The embedding at explicit positions is embed_fwd with a position array (fused_ops.cu).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <stdexcept>
#include <string>

#include "decode.h"
#include "ptx.cuh"
#include "rope.cuh"

namespace pb {

namespace {

constexpr float LOG2E = 1.4426950408889634f;
constexpr float LN2 = 0.6931471805599453f;
constexpr int DA_STAGES = 4;    // ring depth: tiles in flight per CTA
constexpr int DA_WARPS = 4;
constexpr int DA_TK = DECODE_TILE_KEYS;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffff, v, o);
  return v;
}

// ------------------------------------------------------------------ decode attention
// Grid (B*H, n_split), 128 threads. CTA (bh, s) owns keys [s*per, min((s+1)*per, L)) of row b, head h, where L = lengths[b]
// and per = ceil(L / n_split) rounded up to a tile: the split follows each row's own length, read on the device.
// Warp 0 streams the k and v rows of each tile (dh*2 bytes per key and operand, one cp.async.bulk per lane) into a
// DA_STAGES-deep shared-memory ring, completion counted on a per-stage mbarrier. Each warp scores DA_TK/4 keys of a
// tile (lane = dh/32 dims, butterfly sum) and keeps its own online-softmax state in the log2 domain; the four warps are
// merged at the end. n_split == 1 writes the normalised output; otherwise the unnormalised partial (o, m, l) goes to
// fp32 scratch for decode_combine_kernel.
template <int DH>
__global__ void __launch_bounds__(DA_WARPS * 32) decode_attn_kernel(const __nv_bfloat16* __restrict__ q, long long ldq,
                                                                   const __nv_bfloat16* __restrict__ kv, int s_max, int H,
                                                                   const int* __restrict__ lengths, const float* __restrict__ alibi,
                                                                   float scale_log2, float* __restrict__ part,
                                                                   __nv_bfloat16* __restrict__ out, float* __restrict__ lse) {
  constexpr int VPL = DH / 32;             // dims per lane
  constexpr int KPW = DA_TK / DA_WARPS;    // keys per warp per tile
  constexpr uint32_t ROW_BYTES = DH * 2;
  extern __shared__ __align__(128) uint8_t da_smem[];
  __shared__ uint64_t full[DA_STAGES];
  __shared__ float red_m[DA_WARPS], red_l[DA_WARPS];
  __shared__ float red_o[DA_WARPS][DH];
  const int bh = blockIdx.x, split = blockIdx.y, n_split = gridDim.y;
  const int b = bh / H, h = bh - b * H;
  const int d = H * DH;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int L = min(max(lengths[b], 0), s_max);
  const int per = ((L + n_split - 1) / n_split + DA_TK - 1) / DA_TK * DA_TK;
  const int k0 = min(split * per, L), k1 = min(k0 + per, L);
  const int ntiles = (k1 - k0 + DA_TK - 1) / DA_TK;
  const __nv_bfloat16* kvb = kv + (long long)b * s_max * 2 * d + h * DH;
  auto kst = [&](int s) { return reinterpret_cast<__nv_bfloat16*>(da_smem + s * 2 * DA_TK * ROW_BYTES); };
  auto vst = [&](int s) { return kst(s) + DA_TK * DH; };

  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < DA_STAGES; ++s) mbar_init(&full[s], 1);
    fence_barrier_init();
  }
  __syncthreads();
  auto issue = [&](int t) {   // warp 0: tile t -> stage t % DA_STAGES
    const int s = t % DA_STAGES, first = k0 + t * DA_TK, n = min(DA_TK, k1 - first);
    if (lane == 0) mbar_expect_tx(&full[s], uint32_t(n) * 2u * ROW_BYTES);
    __syncwarp();
    if (lane < n) {
      const __nv_bfloat16* row = kvb + (long long)(first + lane) * 2 * d;
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(kst(s) + lane * DH)),
                   "l"(reinterpret_cast<uint64_t>(row)), "r"(ROW_BYTES), "r"(smem_u32(&full[s]))
                   : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(vst(s) + lane * DH)),
                   "l"(reinterpret_cast<uint64_t>(row + d)), "r"(ROW_BYTES), "r"(smem_u32(&full[s]))
                   : "memory");
    }
  };
  if (warp == 0)
    for (int t = 0; t < min(DA_STAGES, ntiles); ++t) issue(t);

  float qf[VPL];
  {
    const __nv_bfloat16* qr = q + (long long)b * ldq + h * DH + lane * VPL;
#pragma unroll
    for (int v = 0; v < VPL; v += 2) {
      const float2 f = unpack_bf16(*reinterpret_cast<const uint32_t*>(qr + v));
      qf[v] = f.x * scale_log2, qf[v + 1] = f.y * scale_log2;
    }
  }
  const float slope = alibi ? alibi[h] * LOG2E : 0.f;
  float m = -INFINITY, l = 0.f, acc[VPL];
#pragma unroll
  for (int v = 0; v < VPL; ++v) acc[v] = 0.f;

  for (int t = 0; t < ntiles; ++t) {
    const int s = t % DA_STAGES, first = k0 + t * DA_TK, n = min(DA_TK, k1 - first);
    mbar_wait(&full[s], uint32_t((t / DA_STAGES) & 1));
    const __nv_bfloat16* Ks = kst(s);
    const __nv_bfloat16* Vs = vst(s);
    float sc[KPW];
    float mt = -INFINITY;
#pragma unroll
    for (int j = 0; j < KPW; ++j) {
      const int key = warp * KPW + j;
      float dot = 0.f;
      if (key < n) {
        const __nv_bfloat16* kr = Ks + key * DH + lane * VPL;
#pragma unroll
        for (int v = 0; v < VPL; v += 2) {
          const float2 f = unpack_bf16(*reinterpret_cast<const uint32_t*>(kr + v));
          dot = fmaf(qf[v], f.x, fmaf(qf[v + 1], f.y, dot));
        }
      }
      dot = warp_sum(dot);
      sc[j] = key < n ? dot + slope * float(first + key - (L - 1)) : -INFINITY;
      mt = fmaxf(mt, sc[j]);
    }
    if (mt > -INFINITY) {
      const float mn = fmaxf(m, mt);
      const float corr = exp2f(m - mn);   // m = -inf on the first tile: corr = 0 and l, acc are still 0
      l *= corr;
#pragma unroll
      for (int v = 0; v < VPL; ++v) acc[v] *= corr;
#pragma unroll
      for (int j = 0; j < KPW; ++j) {
        const int key = warp * KPW + j;
        if (key < n) {
          const float p = exp2f(sc[j] - mn);
          l += p;
          const __nv_bfloat16* vr = Vs + key * DH + lane * VPL;
#pragma unroll
          for (int v = 0; v < VPL; v += 2) {
            const float2 f = unpack_bf16(*reinterpret_cast<const uint32_t*>(vr + v));
            acc[v] = fmaf(p, f.x, acc[v]), acc[v + 1] = fmaf(p, f.y, acc[v + 1]);
          }
        }
      }
      m = mn;
    }
    __syncthreads();   // every warp is done with stage s before it is refilled
    if (warp == 0 && t + DA_STAGES < ntiles) issue(t + DA_STAGES);
  }

  if (lane == 0) red_m[warp] = m, red_l[warp] = l;
#pragma unroll
  for (int v = 0; v < VPL; ++v) red_o[warp][lane * VPL + v] = acc[v];
  __syncthreads();
  float M = red_m[0];
#pragma unroll
  for (int w = 1; w < DA_WARPS; ++w) M = fmaxf(M, red_m[w]);
  float wt[DA_WARPS], Ls = 0.f;
#pragma unroll
  for (int w = 0; w < DA_WARPS; ++w) {
    wt[w] = red_m[w] > -INFINITY ? exp2f(red_m[w] - M) : 0.f;
    Ls += red_l[w] * wt[w];
  }
  for (int i = threadIdx.x; i < DH; i += blockDim.x) {
    float o = 0.f;
#pragma unroll
    for (int w = 0; w < DA_WARPS; ++w) o += red_o[w][i] * wt[w];
    if (n_split == 1) {
      out[(long long)b * d + h * DH + i] = __float2bfloat16(Ls > 0.f ? o / Ls : 0.f);
    } else {
      part[((long long)bh * n_split + split) * DH + i] = o;
    }
  }
  if (threadIdx.x == 0) {
    if (n_split == 1) {
      if (lse) lse[bh] = Ls > 0.f ? (M + log2f(Ls)) * LN2 : -INFINITY;
    } else {
      float* ml = part + (long long)gridDim.x * n_split * DH + ((long long)bh * n_split + split) * 2;
      ml[0] = M, ml[1] = Ls;
    }
  }
}

// Merge of the n_split partials of one (row, head): grid B*H, one thread per output dim.
__global__ void decode_combine_kernel(const float* __restrict__ part, int BH, int n_split, int H, int DH,
                                      __nv_bfloat16* __restrict__ out, float* __restrict__ lse) {
  const int bh = blockIdx.x, b = bh / H, h = bh - b * H;
  const float* ml = part + (long long)BH * n_split * DH + (long long)bh * n_split * 2;
  float M = -INFINITY;
  for (int s = 0; s < n_split; ++s) M = fmaxf(M, ml[2 * s]);
  float Ls = 0.f;
  for (int s = 0; s < n_split; ++s)
    if (ml[2 * s] > -INFINITY) Ls += ml[2 * s + 1] * exp2f(ml[2 * s] - M);
  for (int i = threadIdx.x; i < DH; i += blockDim.x) {
    float o = 0.f;
    for (int s = 0; s < n_split; ++s)
      if (ml[2 * s] > -INFINITY) o += part[((long long)bh * n_split + s) * DH + i] * exp2f(ml[2 * s] - M);
    out[(long long)b * H * DH + h * DH + i] = __float2bfloat16(Ls > 0.f ? o / Ls : 0.f);
  }
  if (threadIdx.x == 0 && lse) lse[bh] = Ls > 0.f ? (M + log2f(Ls)) * LN2 : -INFINITY;
}

// ------------------------------------------------------------------ KV-cache write (+ RoPE)
// One block per qkv row. rotate: every (q|k, head, 8-pair group) is rotated in place by rope_rotate8 and the rotated k is
// also stored to the cache; the v third is copied as is. Rows whose (b, pos) lies outside the cache are skipped.
__global__ void __launch_bounds__(128) kv_write_kernel(__nv_bfloat16* __restrict__ qkv, long long ldq, __nv_bfloat16* __restrict__ cache,
                                                        int B, int s_max, const int* __restrict__ b_idx, const int* __restrict__ pos,
                                                        const float* __restrict__ cosT, const float* __restrict__ sinT, long long T,
                                                        int H, int dh, int rotate) {
  const int d = H * dh;
  for (long long t = blockIdx.x; t < T; t += gridDim.x) {
    const int b = b_idx[t], p = pos[t];
    if (b < 0 || b >= B || p < 0 || p >= s_max) continue;
    __nv_bfloat16* row = qkv + t * ldq;
    __nv_bfloat16* dst = cache + ((long long)b * s_max + p) * 2 * d;
    if (rotate) {
      const int half = dh / 2, groups = half / 8, n = 2 * H * groups;
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int g = i % groups, r = i / groups, hh = r % H, which = r / H;
        __nv_bfloat16* base = row + which * d + hh * dh + g * 8;
        uint4 a = *reinterpret_cast<const uint4*>(base);
        uint4 c = *reinterpret_cast<const uint4*>(base + half);
        rope_rotate8(a, c, cosT + (long long)p * half + g * 8, sinT + (long long)p * half + g * 8, 0);
        *reinterpret_cast<uint4*>(base) = a;
        *reinterpret_cast<uint4*>(base + half) = c;
        if (which == 1) {
          *reinterpret_cast<uint4*>(dst + hh * dh + g * 8) = a;
          *reinterpret_cast<uint4*>(dst + hh * dh + g * 8 + half) = c;
        }
      }
      for (int i = threadIdx.x; i < d / 8; i += blockDim.x)
        reinterpret_cast<uint4*>(dst + d)[i] = reinterpret_cast<const uint4*>(row + 2 * d)[i];
    } else {
      for (int i = threadIdx.x; i < 2 * d / 8; i += blockDim.x)
        reinterpret_cast<uint4*>(dst)[i] = reinterpret_cast<const uint4*>(row + d)[i];
    }
  }
}

// ------------------------------------------------------------------ row argmax
// One block per row; ties resolve to the lowest index (strictly-greater updates in index order, then index-aware merges).
__global__ void __launch_bounds__(256) argmax_rows_kernel(const __nv_bfloat16* __restrict__ logits, long long ld, int V,
                                                           int64_t* __restrict__ out) {
  __shared__ float sv[8];
  __shared__ int si[8];
  const __nv_bfloat16* r = logits + (long long)blockIdx.x * ld;
  float best = -INFINITY;
  int bi = V;
  const bool vec = (V % 8 == 0) && (ld % 8 == 0) && ((reinterpret_cast<uintptr_t>(logits) & 15) == 0);
  if (vec) {
    for (int i = threadIdx.x; i < V / 8; i += blockDim.x) {
      const uint4 u = reinterpret_cast<const uint4*>(r)[i];
      const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float2 f = unpack_bf16(w[k]);
        if (f.x > best) best = f.x, bi = i * 8 + 2 * k;
        if (f.y > best) best = f.y, bi = i * 8 + 2 * k + 1;
      }
    }
  } else {
    for (int i = threadIdx.x; i < V; i += blockDim.x) {
      const float f = __bfloat162float(r[i]);
      if (f > best) best = f, bi = i;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffff, best, o);
    const int oi = __shfl_xor_sync(0xffffffff, bi, o);
    if (ov > best || (ov == best && oi < bi)) best = ov, bi = oi;
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) sv[w] = best, si[w] = bi;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < int(blockDim.x >> 5); ++i)
      if (sv[i] > best || (sv[i] == best && si[i] < bi)) best = sv[i], bi = si[i];
    out[blockIdx.x] = bi < V ? bi : 0;   // a row with no ordered value (all NaN / -inf) yields 0
  }
}

void check_launch(const char* name) {
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) throw std::runtime_error(std::string(name) + " launch: " + cudaGetErrorString(e));
}

template <int DH>
void launch_attn(const void* q, long long ldq, const void* kv, int B, int s_max, int H, const int* lengths, const float* alibi,
                 float scale_log2, int n_split, float* scratch, void* out, float* lse, cudaStream_t st) {
  constexpr int smem = DA_STAGES * 2 * DA_TK * DH * 2;
  static bool configured = false;
  if (!configured) {
    const cudaError_t e = cudaFuncSetAttribute(decode_attn_kernel<DH>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) throw std::runtime_error(std::string("decode_attention smem attr: ") + cudaGetErrorString(e));
    configured = true;
  }
  decode_attn_kernel<DH><<<dim3(B * H, n_split), DA_WARPS * 32, smem, st>>>(
      (const __nv_bfloat16*)q, ldq, (const __nv_bfloat16*)kv, s_max, H, lengths, alibi, scale_log2, scratch, (__nv_bfloat16*)out,
      lse);
  check_launch("decode_attention");
}

}  // namespace

int decode_attention_splits(int BH, int s_max, int num_sms) {
  const int max_split = std::max(1, (s_max + DA_TK - 1) / DA_TK);
  const int want = (8 * std::max(num_sms, 1) + BH - 1) / std::max(BH, 1);
  return std::max(1, std::min(want, max_split));
}

int decode_attention_launch(const void* q, long long ldq, const void* kv, int B, int s_max, int H, int dh, const int* lengths,
                            const float* alibi, float scale, int n_split, float* scratch, void* out, float* lse, cudaStream_t st) {
  if (B <= 0) return 0;
  if (n_split < 1 || (n_split > 1 && !scratch)) throw std::runtime_error("decode_attention: n_split > 1 needs the fp32 scratch");
  const float sl = scale * LOG2E;
  if (dh == 64) launch_attn<64>(q, ldq, kv, B, s_max, H, lengths, alibi, sl, n_split, scratch, out, lse, st);
  else if (dh == 128) launch_attn<128>(q, ldq, kv, B, s_max, H, lengths, alibi, sl, n_split, scratch, out, lse, st);
  else throw std::runtime_error("decode_attention: d_head must be 64 or 128");
  if (n_split == 1) return 1;
  decode_combine_kernel<<<B * H, dh, 0, st>>>(scratch, B * H, n_split, H, dh, (__nv_bfloat16*)out, lse);
  check_launch("decode_combine");
  return 2;
}

void kv_write_launch(void* qkv, long long ldq, void* cache, int B, int s_max, const int* b_idx, const int* pos, const float* cosT,
                     const float* sinT, long long T, int H, int dh, bool rotate, cudaStream_t st) {
  if (T <= 0) return;
  if (dh % 16) throw std::runtime_error("kv_write: d_head must be a multiple of 16");
  const int blocks = int(std::min<long long>(T, 148 * 16));
  kv_write_kernel<<<blocks, 128, 0, st>>>((__nv_bfloat16*)qkv, ldq, (__nv_bfloat16*)cache, B, s_max, b_idx, pos, cosT, sinT, T, H, dh,
                                          rotate ? 1 : 0);
  check_launch("kv_write");
}

void argmax_rows_launch(const void* logits, long long ld, long long R, int V, int64_t* out, cudaStream_t st) {
  if (R <= 0) return;
  argmax_rows_kernel<<<int(R), 256, 0, st>>>((const __nv_bfloat16*)logits, ld, V, out);
  check_launch("argmax_rows");
}

}  // namespace pb
