// Causal flash attention for sm_100a on tcgen05 tensor cores with TMEM-resident S / P / O.
//
// Forward (attn_fwd_kernel<DH>): one CTA = one (batch, head, 128-query tile).
//   warp 4 : TMA producer  — Q once, then a 2-stage ring of K / V tiles straight out of the fused
//            [B*S, 3*d] QKV projection output (no head split / transpose copies)
//   warp 5 : MMA issuer    — S = Q K^T (SS, both K-major) into TMEM; O += P V with P read FROM TMEM
//            (TS form) and V consumed MN-major as stored
//   warps 0-3: softmax      — one thread per query row (TMEM lane): tcgen05.ld S, online max/sum in
//            the log2 domain, P written back to TMEM as packed bf16 (tcgen05.st), lazy O rescale
// For d_head = 64 a CTA needs 256 TMEM columns and 80 KiB smem, so two CTAs share an SM and one CTA's
// softmax overlaps the other's MMAs.
//
// Backward (attn_bwd_kernel<64>): one CTA = one (batch, head, 128-key tile) holding K_j, V_j in smem and
// dK_j, dV_j in TMEM; loops over the query tiles i >= j: S = Q K^T and dP = dO V^T (SS), P / dS computed by
// the row threads and staged in smem ONCE in a layout that is simultaneously K-major (for dQ = dS K) and
// MN-major (for dV += P^T dO, dK += dS^T Q); dQ partial tiles leave through TMA reduce-add (fp32).
//
// Replaces flash-attn 2.x (mma.sync/cp.async) the reference calls through llm-foundry (SURVEY §2.5 K4).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <stdexcept>
#include <string>
#include <type_traits>

#include "attention_tcgen05.h"
#include "gemm_tcgen05.h"
#include "ptx.cuh"
#include "rope.cuh"

namespace pb {

namespace {

constexpr int BQ = 128, BKV = 128;
constexpr float LOG2E = 1.4426950408889634f;
constexpr float LN2 = 0.6931471805599453f;

// ======================================================================================= forward
// Persistent kernel: one CTA per SM walks a list of (batch*head, query tile) work items; the TMA, MMA and softmax
// pipelines run ACROSS item boundaries (a one-tile-per-CTA grid measured 3.9 us of prologue/epilogue per CTA against
// 0.89 us per KV tile — a third of the run time at S = 2048).
//   warp 4*NS   : TMA producer  — Q (double-buffered), K ring, V ring
//   warp 4*NS+1 : MMA issuer    — the KV tiles of all items form ONE stream n = 0, 1, 2, ...: S_n = Q K_n^T (SS) goes into
//             S buffer (n & 1) one tile AHEAD of the softmax, O += P_n V_n (TS, P read from TMEM) follows softmax_n.
//             The whole warp walks the loop (uniform operands), one elected lane issues (see gemm_tcgen05.cu).
//   warps 0 .. 4*NS-1: softmax — the NS warps w, w+4, ... (same SM sub-partition, same 32 TMEM lanes) split a query
//             row's 128 key columns NS ways, so every sub-partition has NS warps to interleave (one warp alone reaches
//             ~0.6 IPC; with two the MUFU pipe measured 54 % busy, the rest fixed-latency dependency stalls). The half row is streamed from TMEM in 32-column chunks (next chunk in
//             flight while the current one is exponentiated), only packed bf16 P stays in registers.
//             Exponentials are taken OPTIMISTICALLY against the running reference max; the tile max is tracked on the
//             side and only if a row outgrew the reference by > 2^8 (or on an item's first tile) the tile is redone
//             against the new max (S is still intact in TMEM); the two halves of a row agree on the tile max through
//             smem and a 64-thread named barrier AFTER the exponentials. The epilogue of item i (O / l -> bf16 -> global) is
//             deferred until after the first tile of item i+1, so its wait for the last P V never stalls the stream
//             (O is double-buffered by item parity).
template <int DH>
struct FwdCfg {
  static constexpr int CH = DH / 64;              // 64-column swizzle chunks per tile
  static constexpr int TILE = 128 * 128 * CH;     // bytes of one [128 x DH] bf16 tile
  static constexpr int QBUF = 2;
  static constexpr int KST = (DH == 64) ? 4 : 2;
  static constexpr int VST = (DH == 64) ? 4 : 2;
  static constexpr int AUX = 9216;                // barriers (512 B) + row max / row sum exchange (4 slots x NS<=4 x 128 floats)
  static constexpr int SMEM = TILE * (QBUF + KST + VST) + AUX + 1024;
  // two S buffers (128 fp32 columns each); P_n (packed bf16, 64 columns) aliases the head of S_n; two O accumulators
  static constexpr int COL_S = 0, COL_O = 256;
  static constexpr int TMEM_COLS = 512;
  static_assert(COL_O + 2 * DH <= 512, "TMEM budget");
  static_assert(SMEM <= 232448, "smem budget");
};

// work item k -> (bh, qt). The q-tiles of one (batch, head) are adjacent in k so that the CTAs working on them at the same
// time share K/V through L2; the rotation by bh spreads the causal tile weights evenly over the CTAs of a static
// round-robin schedule (grid % n_qt would otherwise pin every CTA to a few tile sizes).
struct FwdSched {
  int n_qt, n_items, cyc_rounds, grid;
  __device__ __forceinline__ void decode(int k, int& bh, int& qt) const {
    bh = k / n_qt;
    const int slot = k - bh * n_qt;
    const int shift = (bh * n_qt / grid) / cyc_rounds;
    qt = n_qt - 1 - (slot + shift) % n_qt;
  }
};

// 2^x on the FMA / integer pipes (no MUFU): round-to-nearest split x = n + f, |f| <= 0.5, a degree-3 minimax polynomial for 2^f
// (max relative error 7.5e-5, far below the bf16 rounding of P) and n added into the exponent field. The forward softmax is
// bound by the 16 exp2 / clk / SM of the MUFU pipe while the FMA pipe idles: every POLY-th pair of a row goes this way.
__device__ __forceinline__ float exp2_fma(float x) {
  x = fmaxf(x, -126.0f);                        // masked (-inf) scores end as 2^-126 ~ 0
  const float r = x + 12582912.0f;              // 1.5 * 2^23: the integer part lands in the low mantissa bits
  const float f = x - (r - 12582912.0f);
  float p = fmaf(f, 0.05517132207751274f, 0.24261054396629333f);
  p = fmaf(p, f, 0.6932609677314758f);
  p = fmaf(p, f, 0.9999281167984009f);
  return __int_as_float(__float_as_int(p) + (__float_as_int(r) << 23));
}

template <int DH, int NS, bool ALIBI, int POLY>
__global__ void __launch_bounds__((4 * NS + 2) * 32, 1)
attn_fwd_kernel(const __grid_constant__ CUtensorMap tmQKV, __nv_bfloat16* __restrict__ out, float* __restrict__ lse, int S, int H,
                float scale, int causal, const FwdSched sched, const float* __restrict__ alibi_slopes) {
  using C = FwdCfg<DH>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;                             // [QBUF]
  uint8_t* sK = sQ + C::QBUF * C::TILE;           // [KST]
  uint8_t* sV = sK + C::KST * C::TILE;            // [VST]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + C::VST * C::TILE);
  uint64_t* q_full = bars;                        // [2]
  uint64_t* q_empty = bars + 2;                   // [2]
  uint64_t* k_full = bars + 4;                    // [4]
  uint64_t* k_empty = bars + 8;                   // [4]
  uint64_t* v_full = bars + 12;                   // [4]
  uint64_t* v_empty = bars + 16;                  // [4]
  uint64_t* s_full = bars + 20;                   // [2]  S_n landed in buffer n & 1
  uint64_t* p_ready = bars + 22;                  // [2]  P_n stored (128 arrivals)
  uint64_t* pv_done = bars + 24;                  // P V_n retired (per tile; only waited on a rescale)
  uint64_t* o_final = bars + 25;                  // [2]  all P V of an item (by item parity) retired
  uint64_t* o_free = bars + 27;                   // [2]  O buffer drained by the epilogue (256 arrivals)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 40);   // own line, away from the mbarrier words
  float* xch = reinterpret_cast<float*>(bars + 64);    // [4 slots][NS parts][128 rows]
  constexpr int W_TMA = 4 * NS, W_MMA = 4 * NS + 1, COLS = 128 / NS;

  const int warp = __shfl_sync(0xffffffff, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const int d_model = H * DH;
  const int n_items = sched.n_items;
  auto nkv_of = [&](int k) {
    int bh, qt;
    sched.decode(k, bh, qt);
    return causal ? qt + 1 : S / BKV;
  };

  if (warp == W_TMA && lane == 0) {
    prefetch_tmap(&tmQKV);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&q_full[s], 1);
      mbar_init(&q_empty[s], 1);
      mbar_init(&s_full[s], 1);
      mbar_init(&p_ready[s], 128 * NS);
      mbar_init(&o_free[s], 128 * NS);
      mbar_init(&o_final[s], 1);
    }
    for (int s = 0; s < 4; ++s) {
      mbar_init(&k_full[s], 1);
      mbar_init(&k_empty[s], 1);
      mbar_init(&v_full[s], 1);
      mbar_init(&v_empty[s], 1);
    }
    mbar_init(pv_done, 1);
    fence_barrier_init();
  }
  if (warp == W_MMA) tmem_alloc<C::TMEM_COLS>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == W_TMA) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int it = 0, kc = 0, vc = 0;
      for (int k = blockIdx.x; k < n_items; k += gridDim.x, ++it) {
        int bh, qt;
        sched.decode(k, bh, qt);
        const int b = bh / H, h = bh - b * H;
        const int n_kv = causal ? qt + 1 : S / BKV;
        const int qb = it & 1;
        mbar_wait(&q_empty[qb], ((it >> 1) & 1) ^ 1);
        mbar_expect_tx(&q_full[qb], C::TILE);
#pragma unroll
        for (int c = 0; c < C::CH; ++c) tma_load_2d(sQ + qb * C::TILE + c * 16384, &tmQKV, &q_full[qb], h * DH + c * 64, b * S + qt * BQ);
        for (int j = 0; j < n_kv; ++j) {
          const int ks = kc % C::KST;
          mbar_wait(&k_empty[ks], ((kc / C::KST) & 1) ^ 1);
          mbar_expect_tx(&k_full[ks], C::TILE);
#pragma unroll
          for (int c = 0; c < C::CH; ++c)
            tma_load_2d(sK + ks * C::TILE + c * 16384, &tmQKV, &k_full[ks], d_model + h * DH + c * 64, b * S + j * BKV);
          ++kc;
          const int vs = vc % C::VST;
          mbar_wait(&v_empty[vs], ((vc / C::VST) & 1) ^ 1);
          mbar_expect_tx(&v_full[vs], C::TILE);
#pragma unroll
          for (int c = 0; c < C::CH; ++c)
            tma_load_2d(sV + vs * C::TILE + c * 16384, &tmQKV, &v_full[vs], 2 * d_model + h * DH + c * 64, b * S + j * BKV);
          ++vc;
        }
      }
    }
  } else if (warp == W_MMA) {
    // ------------------------------------------------------------------ MMA issuer (whole warp, elected lane issues)
    constexpr uint32_t idesc_s = make_idesc_bf16(BQ, BKV, 0, 0);
    constexpr uint32_t idesc_o = make_idesc_bf16(BQ, DH, 0, 1);
    struct Cur {
      int k, it, j, n_kv;
    };
    auto advance = [&](Cur& c) {
      if (++c.j == c.n_kv) {
        c.k += gridDim.x;
        ++c.it;
        c.j = 0;
        c.n_kv = c.k < n_items ? nkv_of(c.k) : 0;
      }
    };
    int kc = 0, vc = 0, ns = 0, n = 0;
    auto issue_s = [&](const Cur& c) {  // S_ns = Q K^T into S buffer (ns & 1)
      const int qb = c.it & 1;
      if (c.j == 0) mbar_wait(&q_full[qb], (c.it >> 1) & 1);
      const int ks = kc % C::KST;
      mbar_wait(&k_full[ks], (kc / C::KST) & 1);
      tc_fence_after();
      const uint32_t d_col = tmem + C::COL_S + (ns & 1) * 128;
      const uint32_t qd = smem_desc_lo(smem_u32(sQ + qb * C::TILE), 16);
      const uint32_t kd = smem_desc_lo(smem_u32(sK + ks * C::TILE), 16);
#pragma unroll
      for (int kk = 0; kk < DH / 16; ++kk) {
        const uint32_t off = uint32_t(((kk >> 2) * 16384 + (kk & 3) * 32) >> 4);  // descriptor address field is addr >> 4
        if (elect_one()) tc_mma_f16_ss_lo(d_col, qd + off, kd + off, idesc_s, kk != 0);
      }
      if (elect_one()) {
        tc_commit(&s_full[ns & 1]);
        tc_commit(&k_empty[ks]);
        if (c.j == c.n_kv - 1) tc_commit(&q_empty[qb]);  // last read of this Q buffer
      }
      __syncwarp();
      ++kc;
      ++ns;
    };
    Cur nx{int(blockIdx.x), 0, 0, 0};
    nx.n_kv = nx.k < n_items ? nkv_of(nx.k) : 0;
    Cur cu = nx;
    if (nx.k < n_items) {
      issue_s(nx);
      advance(nx);
    }
    while (cu.k < n_items) {
      // S_{n+1} (possibly the next item's first tile) goes first: it runs while the row threads work on S_n. Its buffer
      // held P_{n-1}, consumed by P V_{n-1} issued in the previous iteration (in-order pipe).
      if (nx.k < n_items) {
        issue_s(nx);
        advance(nx);
      }
      const int ob = cu.it & 1;
      if (cu.j == 0) {  // the O buffer of this item parity must have been drained by the epilogue two items ago
        mbar_wait(&o_free[ob], ((cu.it >> 1) & 1) ^ 1);
      }
      const int vs = vc % C::VST;
      mbar_wait(&p_ready[n & 1], (n >> 1) & 1);
      mbar_wait(&v_full[vs], (vc / C::VST) & 1);
      tc_fence_after();
      const uint32_t o_col = tmem + C::COL_O + ob * DH;
      const uint32_t p_col = tmem + C::COL_S + (n & 1) * 128;
      const uint32_t vd = smem_desc_lo(smem_u32(sV + vs * C::TILE), 16384);
#pragma unroll
      for (int kk = 0; kk < BKV / 16; ++kk) {
        // every column part of a row packs its probabilities over the head of its OWN S columns: keys [16 kk, 16 kk + 16)
        // belong to part (16 kk) / COLS and sit at packed column ((16 kk) % COLS) / 2 inside it
        if (elect_one())
          tc_mma_f16_ts_lo(o_col, p_col + ((kk * 16) / COLS) * COLS + ((kk * 16) % COLS) / 2, vd + uint32_t((kk * 2048) >> 4), idesc_o,
                           (cu.j > 0 || kk != 0) ? 1u : 0u);
      }
      if (elect_one()) {
        tc_commit(&v_empty[vs]);
        tc_commit(pv_done);
        if (cu.j == cu.n_kv - 1) tc_commit(&o_final[ob]);
      }
      __syncwarp();
      ++vc;
      ++n;
      advance(cu);
    }
  } else {
    // ------------------------------------------------------------------ softmax rows (warps 0 .. 4*NS-1)
    const int part = warp >> 2;                         // which COLS key columns of the row
    const int w4 = warp & 3;
    const int row = w4 * 32 + lane;                     // query row inside the tile == TMEM lane
    const uint32_t tl = tmem + (uint32_t(w4 * 32) << 16);
    const float sc = scale * LOG2E;
    constexpr int OC = DH / (16 * NS);                  // 16-column O chunks per part
    int n = 0;                                          // KV tiles processed (stream index)
    struct Pend {
      int valid, b, h, qt, it;
      float m, l;
    } pend{0, 0, 0, 0, 0, 0.f, 0.f};
    // combine a per-thread value over the NS column parts of this row (32*NS-thread named barrier)
    auto row_max = [&](float mine, int slot) -> float {
      float* xb = xch + slot * (NS * 128);
      xb[part * 128 + row] = mine;
      named_bar_sync(2 + w4, 32 * NS);
      float v = mine;
#pragma unroll
      for (int o = 1; o < NS; ++o) v = fmaxf(v, xb[((part + o) % NS) * 128 + row]);
      return v;
    };
    auto row_sum = [&](float mine, int slot) -> float {
      float* xb = xch + slot * (NS * 128);
      xb[part * 128 + row] = mine;
      named_bar_sync(2 + w4, 32 * NS);
      float v = 0.f;
#pragma unroll
      for (int o = 0; o < NS; ++o) v += xb[o * 128 + row];   // same order in every part: bit-identical totals
      return v;
    };
    auto epilogue = [&](const Pend& e) {  // O / l -> bf16 -> global (DH/NS columns per part); lse
      // slots 2,3 of the exchange area: never used by the per-tile max exchange (slots 0,1)
      const float l_tot = row_sum(e.l, 2 + (e.it & 1));
      // one barrier per item parity: the epilogue of item i runs after the first tile of item i+1, whose LAST P V may
      // retire (single-tile items) before a slow thread gets here - a shared barrier could then alias two phases
      mbar_wait(&o_final[e.it & 1], (e.it >> 1) & 1);
      tc_fence_after();
      const float inv_l = 1.0f / l_tot;
      __nv_bfloat16* orow = out + (long long)(e.b * S + e.qt * BQ + row) * d_model + e.h * DH;
      const uint32_t to = tl + C::COL_O + (e.it & 1) * DH;
#pragma unroll
      for (int c = part * OC; c < (part + 1) * OC; ++c) {
        uint32_t r[16];
        tmem_ld_32x16(to + c * 16, r);
        tmem_ld_wait();
#pragma unroll
        for (int t = 0; t < 16; t += 8) {
          uint4 o;
          o.x = pack_bf16(__uint_as_float(r[t]) * inv_l, __uint_as_float(r[t + 1]) * inv_l);
          o.y = pack_bf16(__uint_as_float(r[t + 2]) * inv_l, __uint_as_float(r[t + 3]) * inv_l);
          o.z = pack_bf16(__uint_as_float(r[t + 4]) * inv_l, __uint_as_float(r[t + 5]) * inv_l);
          o.w = pack_bf16(__uint_as_float(r[t + 6]) * inv_l, __uint_as_float(r[t + 7]) * inv_l);
          *reinterpret_cast<uint4*>(orow + c * 16 + t) = o;
        }
      }
      if (part == 0) lse[((long long)e.b * H + e.h) * S + e.qt * BQ + row] = e.m * LN2 + __logf(l_tot);
      tc_fence_before();
      mbar_arrive(&o_free[e.it & 1]);
    };
    int it = 0;
    for (int k = blockIdx.x; k < n_items; k += gridDim.x, ++it) {
      int bh, qt;
      sched.decode(k, bh, qt);
      const int b = bh / H, h = bh - b * H;
      const int n_kv = causal ? qt + 1 : S / BKV;
      const uint32_t to = tl + C::COL_O + (it & 1) * DH;
      float m = -INFINITY, l = 0.f;                     // l = partial row sum over this thread's COLS columns
      // ALiBi (attn_config.alibi): score += slope_h * (key - query) (<= 0 for visible keys), folded into the exponent FMA
      const float slope2 = ALIBI ? alibi_slopes[h] * LOG2E : 0.f;
      auto tile = [&](int j, auto diag_tag) {
        constexpr bool DIAG = decltype(diag_tag)::value;
        // key index of this thread's first column minus its query index (ALiBi distance of column 0 of the part)
        const float dist0 = float(j * BKV + part * COLS - (qt * BQ + row));
        const uint32_t ts = tl + C::COL_S + (n & 1) * 128 + part * COLS;   // this thread's S columns; P goes over their head
        mbar_wait(&s_full[n & 1], (n >> 1) & 1);
        tc_fence_after();
        uint32_t pk[COLS / 2];
        float mx = -INFINITY, rs0 = 0.f, rs1 = 0.f;
        auto sweep = [&](auto&& body) {   // body(chunk index, 32 raw S values); with two chunks the second is in flight during the first
          uint32_t ra[32];
          tmem_ld_32x32(ts, ra);
          tmem_ld_wait();
          if constexpr (COLS == 64) {
            uint32_t rb[32];
            tmem_ld_32x32(ts + 32, rb);
            body(0, ra);
            tmem_ld_wait();
            body(1, rb);
          } else {
            body(0, ra);
          }
        };
        auto masked = [&](const uint32_t (&r)[32], int cc, int t) -> float {
          float v = __uint_as_float(r[t]);
          if (DIAG && part * COLS + cc * 32 + t > row) v = -INFINITY;   // causal mask: columns beyond this row
          return v;
        };
        // scaled (log2-domain) score of element t of chunk cc, ALiBi bias included
        auto score = [&](const uint32_t (&r)[32], int cc, int t) -> float {
          const float v = masked(r, cc, t) * sc;
          return ALIBI ? fmaf(slope2, dist0 + float(cc * 32 + t), v) : v;
        };
        auto exp_pass = [&](float m_ref) {
          rs0 = 0.f, rs1 = 0.f;
          if constexpr (POLY == 16 && !ALIBI) {
            // packed variant: the scale-subtract and the row sum of a pair issue as ONE FFMA2 / FADD2 each (7 instead of 9 issue
            // slots per pair; the softmax warps are issue / latency bound, not MUFU bound)
            const float2 scv = make_float2(sc, sc), mneg = make_float2(-m_ref, -m_ref);
            float2 rs = make_float2(0.f, 0.f);
            sweep([&](int cc, const uint32_t (&r)[32]) {
              float cm0 = -INFINITY, cm1 = -INFINITY;
#pragma unroll
              for (int t = 0; t < 32; t += 2) {
                const float v0 = masked(r, cc, t), v1 = masked(r, cc, t + 1);
                cm0 = fmaxf(cm0, v0);
                cm1 = fmaxf(cm1, v1);
                const float2 x = ffma2(make_float2(v0, v1), scv, mneg);
                const float2 p = make_float2(exp2f(x.x), exp2f(x.y));
                rs = fadd2(rs, p);
                pk[cc * 16 + (t >> 1)] = pack_bf16(p.x, p.y);
              }
              mx = fmaxf(mx, fmaxf(cm0, cm1));
            });
            rs0 = rs.x, rs1 = rs.y;
            return;
          }
          sweep([&](int cc, const uint32_t (&r)[32]) {
            float cm0 = -INFINITY, cm1 = -INFINITY;
#pragma unroll
            for (int t = 0; t < 32; t += 2) {
              float p0, p1, x0, x1;
              if (ALIBI) {
                const float y0 = score(r, cc, t), y1 = score(r, cc, t + 1);
                cm0 = fmaxf(cm0, y0);
                cm1 = fmaxf(cm1, y1);
                x0 = y0 - m_ref, x1 = y1 - m_ref;
              } else {
                const float v0 = masked(r, cc, t), v1 = masked(r, cc, t + 1);
                cm0 = fmaxf(cm0, v0);
                cm1 = fmaxf(cm1, v1);
                x0 = fmaf(v0, sc, -m_ref), x1 = fmaf(v1, sc, -m_ref);
              }
              if (POLY > 0 && POLY != 16 && (t >> 1) % (POLY > 0 ? POLY : 1) == (POLY > 0 ? POLY : 1) - 1) {
                p0 = exp2_fma(x0), p1 = exp2_fma(x1);
              } else {
                p0 = exp2f(x0), p1 = exp2f(x1);
              }
              rs0 += p0;
              rs1 += p1;
              pk[cc * 16 + (t >> 1)] = pack_bf16(p0, p1);
            }
            mx = fmaxf(mx, fmaxf(cm0, cm1));
          });
        };
        const bool first = (j == 0);   // no reference max yet
        if (!first) {
          exp_pass(m);
        } else {
          sweep([&](int cc, const uint32_t (&r)[32]) {
            float cm0 = -INFINITY, cm1 = -INFINITY;
#pragma unroll
            for (int t = 0; t < 32; t += 2) {
              cm0 = fmaxf(cm0, ALIBI ? score(r, cc, t) : masked(r, cc, t));
              cm1 = fmaxf(cm1, ALIBI ? score(r, cc, t + 1) : masked(r, cc, t + 1));
            }
            mx = fmaxf(mx, fmaxf(cm0, cm1));
          });
        }
        // all parts of the row now learn the tile max -> identical decisions
        mx = row_max(mx, n & 1);
        const float mxs = ALIBI ? mx : mx * sc;   // the ALiBi path tracks scaled, biased scores
        const bool bump = first || (mxs - m) > 8.0f;
        float alpha = 1.0f;
        const bool redo = __any_sync(0xffffffff, bump);
        if (redo) {
          const float m_new = bump ? fmaxf(m, mxs) : m;
          alpha = bump ? exp2f(m - m_new) : 1.0f;   // 0 on the first tile (m = -inf)
          exp_pass(m_new);
          m = m_new;
        }
#pragma unroll
        for (int cc = 0; cc < COLS / 32; ++cc) {
          asm volatile(
              "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(
                  ts + cc * 16),
              "r"(pk[cc * 16 + 0]), "r"(pk[cc * 16 + 1]), "r"(pk[cc * 16 + 2]), "r"(pk[cc * 16 + 3]), "r"(pk[cc * 16 + 4]),
              "r"(pk[cc * 16 + 5]), "r"(pk[cc * 16 + 6]), "r"(pk[cc * 16 + 7]), "r"(pk[cc * 16 + 8]), "r"(pk[cc * 16 + 9]),
              "r"(pk[cc * 16 + 10]), "r"(pk[cc * 16 + 11]), "r"(pk[cc * 16 + 12]), "r"(pk[cc * 16 + 13]), "r"(pk[cc * 16 + 14]),
              "r"(pk[cc * 16 + 15])
              : "memory");
        }
        l = l * alpha + (rs0 + rs1);
        // rescale the running O (DH/NS columns per part) only when some row of the warp moved its reference max: wait for
        // P V_{n-1} (P V_{n-2} is known retired: it was issued before S_n, so the parity wait cannot alias)
        if (!first && redo) {
          mbar_wait(pv_done, (n - 1) & 1);
          tc_fence_after();
#pragma unroll
          for (int c = part * OC; c < (part + 1) * OC; ++c) {
            uint32_t ro[16];
            tmem_ld_32x16(to + c * 16, ro);
            tmem_ld_wait();
#pragma unroll
            for (int t = 0; t < 16; ++t) ro[t] = __float_as_uint(__uint_as_float(ro[t]) * alpha);
            tmem_st_32x16(to + c * 16, ro);
          }
        }
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(&p_ready[n & 1]);
        ++n;
      };
      const int j_diag = causal ? n_kv - 1 : -1;
      for (int j = 0; j < n_kv; ++j) {
        if (j == j_diag) tile(j, std::true_type{});
        else tile(j, std::false_type{});
        if (pend.valid) {   // the previous item's epilogue, deferred behind this item's first tile
          epilogue(pend);
          pend.valid = 0;
        }
      }
      pend = Pend{1, b, h, qt, it, m, l};
    }
    if (pend.valid) epilogue(pend);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == W_MMA) tmem_dealloc<C::TMEM_COLS>(tmem);
}

// ======================================================================================= backward
// delta[b,h,q] = sum_d dO * O   (row-wise; feeds dS = P * (dP - delta)).  One thread per 8 contiguous elements (16-byte
// loads), DH/8 adjacent lanes form one (row, head) group and reduce with shuffles; the delta store is scattered but tiny.
__global__ void __launch_bounds__(256) attn_bwd_delta_kernel(const __nv_bfloat16* __restrict__ o, const __nv_bfloat16* __restrict__ dout,
                                                              float* __restrict__ delta, int S, int H, int DH, long long rows) {
  const int gl = DH / 8;                                  // lanes per (row, head): 8 for d_head 64, 16 for 128
  const long long n8 = rows * H * gl;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(o) + i);
    const uint4 g = __ldg(reinterpret_cast<const uint4*>(dout) + i);
    const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, gw[4] = {g.x, g.y, g.z, g.w};
    float acc = 0.f;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const float2 fa = unpack_bf16(aw[t]), fg = unpack_bf16(gw[t]);
      acc += fa.x * fg.x + fa.y * fg.y;
    }
    for (int off = gl >> 1; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffff, acc, off);
    if ((i % gl) == 0) {
      const long long rh = i / gl, r = rh / H;
      const int h = int(rh - r * H);
      const long long bb = r / S, sq = r - bb * S;
      delta[(bb * H + h) * S + sq] = acc;
    }
  }
}

// dq_acc (fp32, [B*S, H*DH]) * scale -> bf16 into the q third of dqkv
__global__ void attn_bwd_dq_convert_kernel(const float* __restrict__ dq_acc, __nv_bfloat16* __restrict__ dqkv, long long rows, int d, float scale) {
  const long long n4 = rows * d / 4;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(dq_acc)[i];
    const long long e = i * 4, r = e / d, c = e % d;
    uint2 o;
    o.x = pack_bf16(v.x * scale, v.y * scale), o.y = pack_bf16(v.z * scale, v.w * scale);
    *reinterpret_cast<uint2*>(dqkv + r * 3 * d + c) = o;
  }
}

// d_head = 128 runs the SAME pipeline in NP = 2 passes per (batch*head, key tile): S and dP contract over the full head
// dimension, dV / dK / dQ are formed for one 64-column half of the head per pass (the B operands of those MMAs are simply
// the pass-th 64-column swizzle chunk of the dO / Q / K tiles), so the TMEM plan (448 of 512 columns) is unchanged. The
// price is recomputing S, dP and the exponentials once more, and - the 32 KiB Q / dO / K / V tiles leave no room for
// double buffering - a serialised S/dP -> rows -> dV/dK/dQ chain per tile.
template <int DH_>
struct BwdCfg {
  static constexpr int DH = DH_;
  static constexpr int CH = DH / 64;                        // 64-column swizzle chunks per Q / K / V / dO tile
  static constexpr int NP = CH;                             // passes per item (one 64-column half of the head each)
  static constexpr int TILE = 128 * 128 * CH;               // [128 x DH] bf16
  static constexpr int NKV = (DH == 64) ? 2 : 1;            // K/V buffers (by item parity)
  static constexpr int NST = (DH == 64) ? 2 : 1;            // Q/dO stages (by tile parity)
  static constexpr int PS_TILE = 2 * 128 * 128;             // [128 x 128] bf16 as two 64-col chunks
  static constexpr int DQ_STAGE = 128 * 64 * 4;             // fp32 [128 x 64] staging (two 32-col chunks)
  static constexpr int SMEM = 2 * NKV * TILE /*K,V*/ + 2 * NST * TILE /*Q,dO*/ + 2 * PS_TILE /*P,dS*/ + DQ_STAGE + 256 + 1024;
  static constexpr int COL_S = 0, COL_DP = 128, COL_DV = 256, COL_DK = 320, COL_DQ = 384;   // dQ: two 64-column buffers (tile parity)
  static constexpr int TMEM_COLS = 512;
  static_assert(SMEM <= 232448, "smem budget");
};

// Persistent: one CTA per SM walks (batch*head, key tile) items; the query tiles of ALL its items form one stream
// n = 0, 1, 2, ... through the TMA / MMA / row-thread pipelines (K/V double-buffered by item parity), so the per-CTA
// prologue and the dK/dV epilogue of a one-item-per-CTA grid (measured ~6 us per item against ~1.8 us per query tile)
// overlap the next item's first tiles.
// 320 threads: warps 0-7 = row threads (two per SMSP: warp w and w+4 own the same 32 query rows / TMEM lanes and
// split the 128 key columns 64/64 - no cross-thread exchange is needed because lse and delta are per-row inputs),
// warp 8 = TMA producer, warp 9 = MMA issuer (whole warp, elected lane) + TMEM allocator.
template <int DH_, bool ALIBI>
__global__ void __launch_bounds__(320, 1)
attn_bwd_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmDO, const __grid_constant__ CUtensorMap tmDQ,
                const float* __restrict__ lse, const float* __restrict__ delta, __nv_bfloat16* __restrict__ dqkv, int S, int H, float scale,
                int causal, const FwdSched sched, float* __restrict__ dq_acc, int dq_red, const float* __restrict__ alibi_slopes) {
  using C = BwdCfg<DH_>;
  constexpr int DH = C::DH, NP = C::NP, NKV = C::NKV, NST = C::NST;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sK = smem;                    // [NKV] by item parity
  uint8_t* sV = sK + NKV * C::TILE;      // [NKV]
  uint8_t* sQ = sV + NKV * C::TILE;      // [NST] by tile parity
  uint8_t* sDO = sQ + NST * C::TILE;     // [NST]
  uint8_t* sP = sDO + NST * C::TILE;     // bf16 [128 q][128 kv] as 2 chunks of [128][64]
  uint8_t* sDS = sP + C::PS_TILE;
  uint8_t* sDQ = sDS + C::PS_TILE;       // fp32 staging
  uint64_t* bars = reinterpret_cast<uint64_t*>(sDQ + C::DQ_STAGE);
  uint64_t* kv_full = bars;              // [2] K_j and V_j of item parity
  uint64_t* kv_empty = bars + 2;         // [2]
  uint64_t* qd_full = bars + 4;          // [2] Q_i + dO_i
  uint64_t* qd_empty = bars + 6;         // [2]
  uint64_t* sdp_full = bars + 8;         // S and dP ready
  uint64_t* pds_ready = bars + 9;        // P, dS in smem (256 arrivals)
  uint64_t* dq_full = bars + 10;         // dQ partial tile in TMEM
  uint64_t* dq_free = bars + 11;         // (unused slot)
  uint64_t* mma_done = bars + 12;        // dV/dK/dQ MMAs of the tile retired -> P/dS smem reusable
  uint64_t* final_done = bars + 13;      // all MMAs of an item retired -> dK/dV complete
  uint64_t* acc_free = bars + 14;        // dK/dV accumulators drained by the epilogue (256 arrivals)
  uint64_t* sdp_free = bars + 15;        // S / dP of the tile are in registers (256 arrivals) -> next S / dP may be issued
  uint64_t* dq_free2 = bars + 16;        // [2] dQ TMEM buffer (tile parity) drained (256 arrivals): the dQ MMAs of tile n
                                         // never wait for the drain of tile n-1, only for that of tile n-2
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 24);   // own line, away from the mbarrier words

  const int warp = __shfl_sync(0xffffffff, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const int n_t = S / 128;
  const int d_model = H * DH;
  const int n_items = sched.n_items * NP;
  // item k -> (b, h, key tile jt, first query tile i0, number of query tiles); pass = k % NP
  auto item_of = [&](int k, int& b, int& h, int& jt, int& i0, int& n_it) {
    int bh, w;
    sched.decode(k / NP, bh, w);
    b = bh / H;
    h = bh - b * H;
    jt = n_t - 1 - w;                    // decode() orders by weight w: heavy first == small key tile index
    i0 = causal ? jt : 0;
    n_it = n_t - i0;
  };

  if (warp == 8 && lane == 0) {
    prefetch_tmap(&tmQKV);
    prefetch_tmap(&tmDO);
    prefetch_tmap(&tmDQ);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&kv_full[s], 1);
      mbar_init(&kv_empty[s], 1);
      mbar_init(&qd_full[s], 1);
      mbar_init(&qd_empty[s], 1);
    }
    mbar_init(sdp_full, 1);
    mbar_init(pds_ready, 256);
    mbar_init(dq_full, 1);
    mbar_init(dq_free, 256);
    mbar_init(&dq_free2[0], 256);
    mbar_init(&dq_free2[1], 256);
    mbar_init(mma_done, 1);
    mbar_init(final_done, 1);
    mbar_init(acc_free, 256);
    mbar_init(sdp_free, 256);
    fence_barrier_init();
  }
  if (warp == 9) tmem_alloc<C::TMEM_COLS>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 8) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int it = 0, n = 0;
      for (int k = blockIdx.x; k < n_items; k += gridDim.x, ++it) {
        int b, h, jt, i0, n_it;
        item_of(k, b, h, jt, i0, n_it);
        const int kb = it % NKV;
        mbar_wait(&kv_empty[kb], ((it / NKV) & 1) ^ 1);
        mbar_expect_tx(&kv_full[kb], 2 * C::TILE);
#pragma unroll
        for (int c = 0; c < C::CH; ++c) {
          tma_load_2d(sK + kb * C::TILE + c * 16384, &tmQKV, &kv_full[kb], d_model + h * DH + c * 64, b * S + jt * 128);
          tma_load_2d(sV + kb * C::TILE + c * 16384, &tmQKV, &kv_full[kb], 2 * d_model + h * DH + c * 64, b * S + jt * 128);
        }
        for (int t = 0; t < n_it; ++t, ++n) {
          const int st = n % NST;
          mbar_wait(&qd_empty[st], ((n / NST) & 1) ^ 1);
          mbar_expect_tx(&qd_full[st], 2 * C::TILE);
#pragma unroll
          for (int c = 0; c < C::CH; ++c) {
            tma_load_2d(sQ + st * C::TILE + c * 16384, &tmQKV, &qd_full[st], h * DH + c * 64, b * S + (i0 + t) * 128);
            tma_load_2d(sDO + st * C::TILE + c * 16384, &tmDO, &qd_full[st], h * DH + c * 64, b * S + (i0 + t) * 128);
          }
        }
      }
    }
  } else if (warp == 9) {
    // ------------------------------------------------------------------ MMA issuer (whole warp; elected lane issues)
    constexpr uint32_t idesc_kk = make_idesc_bf16(128, 128, 0, 0);   // S, dP : both K-major, N = 128
    constexpr uint32_t idesc_mm = make_idesc_bf16(128, 64, 1, 1);    // dV, dK: A (P/dS) MN-major, B (dO/Q half) MN-major, N = 64
    constexpr uint32_t idesc_km = make_idesc_bf16(128, 64, 0, 1);    // dQ    : A (dS) K-major, B (K_j half) MN-major
    const uint32_t p_base = smem_u32(sP), ds_base = smem_u32(sDS);
    // descriptor bases; per-k-step offsets are added to the (addr >> 4) field
    const uint32_t pd_m = smem_desc_lo(p_base, 16384), dsd_m = smem_desc_lo(ds_base, 16384);
    const uint32_t dsd_k = smem_desc_lo(ds_base, 16);
    // all stage / item-parity variants up front: nothing but 32-bit adds between the MMAs of a tile
    uint32_t qd_k2[2], dod_k2[2], qd_m2[2], dod_m2[2], kd_k2[2], vd_k2[2], kd_m2[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int qi = i % NST, ki = i % NKV;   // single-buffered variants alias
      qd_k2[i] = smem_desc_lo(smem_u32(sQ + qi * C::TILE), 16), qd_m2[i] = smem_desc_lo(smem_u32(sQ + qi * C::TILE), 16384);
      dod_k2[i] = smem_desc_lo(smem_u32(sDO + qi * C::TILE), 16), dod_m2[i] = smem_desc_lo(smem_u32(sDO + qi * C::TILE), 16384);
      kd_k2[i] = smem_desc_lo(smem_u32(sK + ki * C::TILE), 16), kd_m2[i] = smem_desc_lo(smem_u32(sK + ki * C::TILE), 16384);
      vd_k2[i] = smem_desc_lo(smem_u32(sV + ki * C::TILE), 16);
    }
    struct Cur {
      int k, it, t, n_it;
    };
    auto nit_of = [&](int k) {
      int b, h, jt, i0, n_it;
      item_of(k, b, h, jt, i0, n_it);
      return n_it;
    };
    auto advance = [&](Cur& c) {
      if (++c.t == c.n_it) {
        c.k += gridDim.x;
        ++c.it;
        c.t = 0;
        c.n_it = c.k < n_items ? nit_of(c.k) : 0;
      }
    };
    int ns = 0, n = 0;
    auto issue_sdp = [&](const Cur& c) {  // S = Q K^T ; dP = dO V^T  (contraction over d_head: 4 k-steps per 64-column swizzle chunk)
      const int st = ns % NST, kb = c.it % NKV;
      if (c.t == 0) mbar_wait(&kv_full[kb], (c.it / NKV) & 1);
      mbar_wait(&qd_full[st], (ns / NST) & 1);
      tc_fence_after();
      const uint32_t qd_k = st ? qd_k2[1] : qd_k2[0], dod_k = st ? dod_k2[1] : dod_k2[0];
      const uint32_t kd_k = kb ? kd_k2[1] : kd_k2[0], vd_k = kb ? vd_k2[1] : vd_k2[0];
#pragma unroll
      for (int kk = 0; kk < DH / 16; ++kk) {
        const uint32_t off = uint32_t(((kk >> 2) * 16384 + (kk & 3) * 32) >> 4);
        if (elect_one()) tc_mma_f16_ss_lo(tmem + C::COL_S, qd_k + off, kd_k + off, idesc_kk, kk != 0);
      }
#pragma unroll
      for (int kk = 0; kk < DH / 16; ++kk) {
        const uint32_t off = uint32_t(((kk >> 2) * 16384 + (kk & 3) * 32) >> 4);
        if (elect_one()) tc_mma_f16_ss_lo(tmem + C::COL_DP, dod_k + off, vd_k + off, idesc_kk, kk != 0);
      }
      if (elect_one()) tc_commit(sdp_full);
      __syncwarp();
      ++ns;
    };
    Cur nx{int(blockIdx.x), 0, 0, 0};
    nx.n_it = nx.k < n_items ? nit_of(nx.k) : 0;
    Cur cu = nx;
    if (nx.k < n_items) {
      issue_sdp(nx);
      advance(nx);
    }
    while (cu.k < n_items) {
      const int st = n % NST, kb = cu.it % NKV;
      const uint32_t half = uint32_t(((cu.k % NP) * 16384) >> 4);   // 64-column chunk of dO / Q / K for this pass
      const uint32_t qd_m = (st ? qd_m2[1] : qd_m2[0]) + half, dod_m = (st ? dod_m2[1] : dod_m2[0]) + half;
      const uint32_t kd_m = (kb ? kd_m2[1] : kd_m2[0]) + half;
      // next tile's S / dP (possibly the next item's) are issued as soon as the row threads hold S_n / dP_n in
      // registers: they run on the tensor pipe while the rows are still computing P_n / dS_n. With a single Q/dO stage
      // (d_head 128) the next tile cannot be loaded before this tile's dV / dK retire: S / dP follow them instead.
      mbar_wait(sdp_free, n & 1);
      if (NST > 1 && nx.k < n_items) {
        issue_sdp(nx);
        advance(nx);
      }
      mbar_wait(pds_ready, n & 1);   // P_n / dS_n staged in smem
      if (n >= 2) mbar_wait(&dq_free2[n & 1], ((n >> 1) & 1) ^ 1);
      if (cu.t == 0 && cu.it > 0) mbar_wait(acc_free, (cu.it - 1) & 1);  // previous item's dK / dV drained
      tc_fence_after();
      const uint32_t acc = cu.t != 0;
      // contraction over the 128 query rows of this tile: 8 k-steps, 16 rows (2048 B = 128 descriptor units) each
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {
        // dV[kv, dh] += P^T dO : A = P (MN-major: kv contiguous, 2 chunks of 64 -> LBO 16 KiB), B = dO (MN-major, N = 64)
        if (elect_one()) tc_mma_f16_ss_lo(tmem + C::COL_DV, pd_m + uint32_t(kk * 128), dod_m + uint32_t(kk * 128), idesc_mm, (acc | kk) != 0);
      }
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {
        // dK[kv, dh] += dS^T Q
        if (elect_one()) tc_mma_f16_ss_lo(tmem + C::COL_DK, dsd_m + uint32_t(kk * 128), qd_m + uint32_t(kk * 128), idesc_mm, (acc | kk) != 0);
      }
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {
        // dQ[q, dh] = dS K_j : A = dS K-major (kv contiguous: chunk = kk/4, 32 B per k-step), B = K_j MN-major over kv rows
        if (elect_one())
          tc_mma_f16_ss_lo(tmem + C::COL_DQ + (n & 1) * 64, dsd_k + uint32_t(((kk >> 2) * 16384 + (kk & 3) * 32) >> 4), kd_m + uint32_t(kk * 128), idesc_km,
                           kk != 0);
      }
      if (elect_one()) {
        tc_commit(&qd_empty[st]);
        tc_commit(dq_full);
        tc_commit(mma_done);
        if (cu.t == cu.n_it - 1) {
          tc_commit(final_done);
          tc_commit(&kv_empty[kb]);
        }
      }
      __syncwarp();
      if (NST == 1 && nx.k < n_items) {
        issue_sdp(nx);
        advance(nx);
      }
      ++n;
      advance(cu);
    }
  } else {
    // ------------------------------------------------------------------ row threads (warps 0..7)
    const int half = warp >> 2;                      // which 64 key columns of the row this thread owns
    const int row = (warp & 3) * 32 + lane;
    const uint32_t tl = tmem + (uint32_t((warp & 3) * 32) << 16);
    const float sc = scale * LOG2E;
    const uint32_t swz = row & 7;
    const bool issuer = (threadIdx.x == 0);
    int n = 0;                                       // query tiles processed (stream index)
    struct Prev {
      int valid, b, h, qt;       // coordinates of tile n-1 (its dQ partial is still in TMEM)
      int item_end, jt, it;      // tile n-1 was the last of item `it` (key tile jt): dK/dV epilogue pending
      int pass;                  // which 64-column half of the head this item covers
    } pv{0, 0, 0, 0, 0, 0, 0, 0};
    auto drain_dq = [&](const Prev& p) {  // dQ partial of tile n-1: TMEM -> fp32 smem staging -> TMA reduce-add into dq_acc
      mbar_wait(dq_full, (n - 1) & 1);
      tc_fence_after();
      if (dq_red) {
        // alternative (PB_ATTN_DQ_RED=1): vector reductions straight from registers - no staging, fence or block barrier,
        // but twice as many (16-byte) L2 atomics as the TMA reduce: measured 2.49 vs 1.85 us per query tile -> off by default
        uint32_t r[32];
        tmem_ld_32x32(tl + C::COL_DQ + ((n - 1) & 1) * 64 + half * 32, r);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(&dq_free2[(n - 1) & 1]);
        float* dst = dq_acc + (long long)(p.b * S + p.qt * 128 + row) * d_model + p.h * DH + p.pass * 64 + half * 32;
#pragma unroll
        for (int g = 0; g < 8; ++g)
          asm volatile("red.relaxed.gpu.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + 4 * g), "f"(__uint_as_float(r[4 * g])),
                       "f"(__uint_as_float(r[4 * g + 1])), "f"(__uint_as_float(r[4 * g + 2])), "f"(__uint_as_float(r[4 * g + 3]))
                       : "memory");
        return;
      }
      if (issuer) tma_wait_read<0>();
      named_bar_sync(1, 256);
      {
        const int c = half;  // 32 of the 64 dQ columns per thread
        uint32_t r[32];
        tmem_ld_32x32(tl + C::COL_DQ + ((n - 1) & 1) * 64 + c * 32, r);
        tmem_ld_wait();
        uint8_t* qrow = sDQ + c * 16384 + row * 128;
#pragma unroll
        for (int g = 0; g < 8; ++g)
          *reinterpret_cast<uint4*>(qrow + ((uint32_t(g) ^ swz) << 4)) = make_uint4(r[4 * g], r[4 * g + 1], r[4 * g + 2], r[4 * g + 3]);
      }
      tc_fence_before();
      mbar_arrive(&dq_free2[(n - 1) & 1]);
      fence_proxy_async_smem();
      named_bar_sync(1, 256);
      if (issuer) {
        tma_reduce_add_2d(&tmDQ, sDQ, p.h * DH + p.pass * 64, p.b * S + p.qt * 128);
        tma_reduce_add_2d(&tmDQ, sDQ + 16384, p.h * DH + p.pass * 64 + 32, p.b * S + p.qt * 128);
        tma_commit();
      }
    };
    auto epilogue = [&](const Prev& p) {  // dK (x scale), dV of item p.it -> bf16 -> dqkv
      mbar_wait(final_done, p.it & 1);
      tc_fence_after();
      __nv_bfloat16* krow = dqkv + (long long)(p.b * S + p.jt * 128 + row) * (3 * d_model) + d_model + p.h * DH + p.pass * 64;
      __nv_bfloat16* vrow = krow + d_model;
      const int c = half;
      uint32_t rk[32], rv[32];
      tmem_ld_32x32(tl + C::COL_DK + c * 32, rk);
      tmem_ld_32x32(tl + C::COL_DV + c * 32, rv);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(acc_free);   // values are in registers: the next item's dV / dK MMAs may overwrite the accumulators
#pragma unroll
      for (int e = 0; e < 32; e += 8) {
        uint4 ok, ov;
        ok.x = pack_bf16(__uint_as_float(rk[e]) * scale, __uint_as_float(rk[e + 1]) * scale);
        ok.y = pack_bf16(__uint_as_float(rk[e + 2]) * scale, __uint_as_float(rk[e + 3]) * scale);
        ok.z = pack_bf16(__uint_as_float(rk[e + 4]) * scale, __uint_as_float(rk[e + 5]) * scale);
        ok.w = pack_bf16(__uint_as_float(rk[e + 6]) * scale, __uint_as_float(rk[e + 7]) * scale);
        ov.x = pack_bf16(__uint_as_float(rv[e]), __uint_as_float(rv[e + 1]));
        ov.y = pack_bf16(__uint_as_float(rv[e + 2]), __uint_as_float(rv[e + 3]));
        ov.z = pack_bf16(__uint_as_float(rv[e + 4]), __uint_as_float(rv[e + 5]));
        ov.w = pack_bf16(__uint_as_float(rv[e + 6]), __uint_as_float(rv[e + 7]));
        *reinterpret_cast<uint4*>(krow + c * 32 + e) = ok;
        *reinterpret_cast<uint4*>(vrow + c * 32 + e) = ov;
      }
    };
    int it = 0;
    for (int k = blockIdx.x; k < n_items; k += gridDim.x, ++it) {
      int b, h, jt, i0, n_it;
      item_of(k, b, h, jt, i0, n_it);
      float nx_lse, nx_dl;
      {
        const long long g0 = (long long)(b * H + h) * S + i0 * 128 + row;
        nx_lse = lse[g0];
        nx_dl = delta[g0];
      }
      const float slope2 = ALIBI ? alibi_slopes[h] * LOG2E : 0.f;
      auto row_tile = [&](int t, auto diag_tag) {
        constexpr bool DIAG = decltype(diag_tag)::value;
        const int qt = i0 + t;
        // ALiBi distance (key - query) of this thread's first column; slope2 == 0 leaves the exponent untouched
        const float bias0 = slope2 * float(jt * 128 + half * 64 - (qt * 128 + row)) - nx_lse * LOG2E;
        const float lse2 = nx_lse * LOG2E;   // this tile's row statistics were fetched one tile ahead
        const float dl = nx_dl;
        mbar_wait(sdp_full, n & 1);
        tc_fence_after();
        uint32_t pk[32], dk[32];  // packed bf16 P and dS of this thread's 64 columns, kept in registers
        uint32_t rs2[2][32], rp2[2][32];
        float pf[64];             // fp32 probabilities until dS is formed
        // S first; the dP loads are in flight while the exponentials run (a TMEM x32 round trip is ~80 clk per warp)
        tmem_ld_32x32(tl + C::COL_S + (half * 2) * 32, rs2[0]);
        tmem_ld_32x32(tl + C::COL_S + (half * 2 + 1) * 32, rs2[1]);
        tmem_ld_wait();
        tmem_ld_32x32(tl + C::COL_DP + (half * 2) * 32, rp2[0]);
        tmem_ld_32x32(tl + C::COL_DP + (half * 2 + 1) * 32, rp2[1]);
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          const int c = half * 2 + cc;  // 32-column block of the row
#pragma unroll
          for (int e = 0; e < 32; e += 2) {
            float p0, p1;
            if (ALIBI) {   // score + slope * (key - query) - lse
              p0 = exp2f(fmaf(__uint_as_float(rs2[cc][e]), sc, fmaf(slope2, float(cc * 32 + e), bias0)));
              p1 = exp2f(fmaf(__uint_as_float(rs2[cc][e + 1]), sc, fmaf(slope2, float(cc * 32 + e + 1), bias0)));
            } else {
              p0 = exp2f(fmaf(__uint_as_float(rs2[cc][e]), sc, -lse2));
              p1 = exp2f(fmaf(__uint_as_float(rs2[cc][e + 1]), sc, -lse2));
            }
            if (DIAG) {
              if (c * 32 + e > row) p0 = 0.f;
              if (c * 32 + e + 1 > row) p1 = 0.f;
            }
            pf[cc * 32 + e] = p0, pf[cc * 32 + e + 1] = p1;
            pk[cc * 16 + (e >> 1)] = pack_bf16(p0, p1);
          }
        }
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(sdp_free);   // S_n / dP_n are in registers: the MMA warp may overwrite them with tile n+1
        // row statistics of the next tile of this item (the first tile of an item fetches its own)
        if (t + 1 < n_it) {
          const long long gnext = (long long)(b * H + h) * S + (qt + 1) * 128 + row;
          nx_lse = lse[gnext];
          nx_dl = delta[gnext];
        }
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
#pragma unroll
          for (int e = 0; e < 32; e += 2) {
            const float s0 = pf[cc * 32 + e] * (__uint_as_float(rp2[cc][e]) - dl);
            const float s1 = pf[cc * 32 + e + 1] * (__uint_as_float(rp2[cc][e + 1]) - dl);
            dk[cc * 16 + (e >> 1)] = pack_bf16(s0, s1);
          }
        }
        // S_n / dP_n are consumed (the MMA warp may overwrite them); the smem staging is reusable once the
        // previous tile's dV / dK / dQ MMAs retired
        if (n > 0) mbar_wait(mma_done, (n - 1) & 1);
        {
          // this thread's 64 columns = swizzle chunk `half` of row `row`: eight 16-byte groups
          uint8_t* prow = sP + half * 16384 + row * 128;
          uint8_t* drow = sDS + half * 16384 + row * 128;
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            const uint32_t slot = (uint32_t(g) ^ swz) << 4;
            *reinterpret_cast<uint4*>(prow + slot) = make_uint4(pk[4 * g], pk[4 * g + 1], pk[4 * g + 2], pk[4 * g + 3]);
            *reinterpret_cast<uint4*>(drow + slot) = make_uint4(dk[4 * g], dk[4 * g + 1], dk[4 * g + 2], dk[4 * g + 3]);
          }
        }
        fence_proxy_async_smem();
        tc_fence_before();
        mbar_arrive(pds_ready);
        // previous tile's dQ partial (and, if it closed an item, that item's dK / dV): overlaps with S/dP of the next
        // tile and dV/dK/dQ of this one on the tensor pipe
        if (pv.valid) {
          drain_dq(pv);
          if (pv.item_end) epilogue(pv);
        }
        pv = Prev{1, b, h, qt, t == n_it - 1, jt, it, k % NP};
        ++n;
      };
      // causal: only the first query tile (qt == jt) touches the diagonal; every other tile runs the mask-free body
      for (int t = 0; t < n_it; ++t) {
        if (causal && t == 0) row_tile(t, std::true_type{});
        else row_tile(t, std::false_type{});
      }
    }
    if (pv.valid) {
      drain_dq(pv);
      epilogue(pv);
    }
    if (issuer) tma_wait_all<0>();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 9) tmem_dealloc<C::TMEM_COLS>(tmem);
}

template <typename K>
void set_smem(K kern, int bytes) {
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) throw std::runtime_error(std::string("attention smem attr: ") + cudaGetErrorString(e));
}

#ifndef PB_ATTN_POLY_DEFAULT
#define PB_ATTN_POLY_DEFAULT 0
#endif

float* g_dq_acc = nullptr;
size_t g_dq_acc_bytes = 0;

}  // namespace

void attention_fwd_launch(const void* qkv, void* out, float* lse, int B, int S, int H, int dh, float scale, bool causal, int num_sms,
                          cudaStream_t st, const float* alibi_slopes) {
  if (S % 128) throw std::runtime_error("photon_b200 attention: sequence length must be a multiple of 128");
  if (dh != 64 && dh != 128) throw std::runtime_error("photon_b200 attention: d_head must be 64 or 128");
  const int d = H * dh;
  CUtensorMap tm = make_tmap_2d(qkv, 2, false, uint64_t(3) * d, uint64_t(B) * S, uint64_t(3) * d * 2, 64, 128);
  FwdSched sched;
  sched.n_qt = S / 128;
  sched.n_items = sched.n_qt * H * B;
  const int sms = num_sms > 0 ? num_sms : 148;
  const int grid = sched.n_items < sms ? sched.n_items : sms;
  sched.grid = grid;
  {  // rounds after which a CTA of the static round-robin has visited every slot class (see FwdSched)
    int a = sched.n_qt, b2 = grid % sched.n_qt;
    while (b2) { const int t = a % b2; a = b2; b2 = t; }
    sched.cyc_rounds = sched.n_qt / a;
  }
  // two column parts per query row = two softmax warps per SM sub-partition (four measured slower: 432 vs 407 us)
  // PB_ATTN_POLY = 4: every 4th pair of exponentials on the FMA pipe (default 0 = all on MUFU). Measured (profiles/attn_exp2_poly.txt):
  // 1/4 -> 0.419 ms, 1/3 -> 0.420, 1/2 -> 0.453 against 0.408 ms with none: the softmax warps are bound by issue slots and
  // fixed-latency dependencies (two warps per scheduler), not by MUFU throughput, so the ~9 extra instructions per element cost
  // more than the MUFU cycles they free. PB_ATTN_POLY = 16: packed FFMA2 / FADD2 in the exponent loop (7 instead of 9 issue slots per
  // pair) -> 0.411 ms, no change: the tile time is set by the MMA -> tcgen05.ld -> softmax -> tcgen05.st -> MMA dependency chain, not
  // by a pipe. Both kept as switches.
  static const int poly = [] { const char* e = std::getenv("PB_ATTN_POLY"); return e ? std::atoi(e) : PB_ATTN_POLY_DEFAULT; }();
#define PB_FWD(DHV, AL, PL)                                                                                           \
  {                                                                                                                   \
    static bool once = (set_smem(attn_fwd_kernel<DHV, 2, AL, PL>, FwdCfg<DHV>::SMEM), true);                           \
    (void)once;                                                                                                       \
    attn_fwd_kernel<DHV, 2, AL, PL><<<grid, 10 * 32, FwdCfg<DHV>::SMEM, st>>>(tm, (__nv_bfloat16*)out, lse, S, H, scale, \
                                                                            causal ? 1 : 0, sched, alibi_slopes);     \
  }
#define PB_FWD_P(DHV, AL)                                                                                             \
  {                                                                                                                   \
    if (poly == 4) PB_FWD(DHV, AL, 4)                                                                                 \
    else if (poly == 16) PB_FWD(DHV, AL, 16)                                                                          \
    else PB_FWD(DHV, AL, 0)                                                                                           \
  }
  if (dh == 64 && !alibi_slopes) PB_FWD_P(64, false)
  else if (dh == 64) PB_FWD_P(64, true)
  else if (!alibi_slopes) PB_FWD_P(128, false)
  else PB_FWD_P(128, true)
#undef PB_FWD_P
#undef PB_FWD
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) throw std::runtime_error(std::string("attention fwd launch: ") + cudaGetErrorString(e));
}

int attention_bwd_launch(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv, float* delta, int B, int S, int H,
                         int dh, float scale, bool causal, int num_sms, cudaStream_t st, const float* alibi_slopes) {
  if (S % 128) throw std::runtime_error("photon_b200 attention: sequence length must be a multiple of 128");
  if (dh != 64 && dh != 128) throw std::runtime_error("photon_b200 attention backward: d_head must be 64 or 128");
  const int d = H * dh;
  const long long rows = (long long)B * S;
  const size_t need = size_t(rows) * d * sizeof(float);
  if (need > g_dq_acc_bytes) {
    if (g_dq_acc) cudaFree(g_dq_acc);
    if (cudaMalloc(&g_dq_acc, need) != cudaSuccess) throw std::runtime_error("attention bwd: dq accumulator allocation failed");
    g_dq_acc_bytes = need;
  }
  cudaMemsetAsync(g_dq_acc, 0, need, st);
  {
    const long long n8 = rows * H * (dh / 8);
    const int blocks = int(std::min<long long>((n8 + 255) / 256, 148 * 16));
    attn_bwd_delta_kernel<<<blocks, 256, 0, st>>>((const __nv_bfloat16*)out, (const __nv_bfloat16*)dout, delta, S, H, dh, rows);
  }
  CUtensorMap tmQKV = make_tmap_2d(qkv, 2, false, uint64_t(3) * d, uint64_t(rows), uint64_t(3) * d * 2, 64, 128);
  CUtensorMap tmDO = make_tmap_2d(dout, 2, false, uint64_t(d), uint64_t(rows), uint64_t(d) * 2, 64, 128);
  CUtensorMap tmDQ = make_tmap_2d(g_dq_acc, 4, true, uint64_t(d), uint64_t(rows), uint64_t(d) * 4, 32, 128);
  FwdSched sched;
  sched.n_qt = S / 128;
  sched.n_items = sched.n_qt * H * B;
  const int sms = num_sms > 0 ? num_sms : 148;
  const int grid = sched.n_items < sms ? sched.n_items : sms;
  sched.grid = grid;
  {
    int a = sched.n_qt, b2 = grid % sched.n_qt;
    while (b2) { const int t = a % b2; a = b2; b2 = t; }
    sched.cyc_rounds = sched.n_qt / a;
  }
  static const int dq_red = [] { const char* e = std::getenv("PB_ATTN_DQ_RED"); return e ? std::atoi(e) : 0; }();
#define PB_BWD(DHV, AL, GRID)                                                                                        \
  {                                                                                                                   \
    static bool once = (set_smem(attn_bwd_kernel<DHV, AL>, BwdCfg<DHV>::SMEM), true);                                  \
    (void)once;                                                                                                       \
    attn_bwd_kernel<DHV, AL><<<GRID, 320, BwdCfg<DHV>::SMEM, st>>>(tmQKV, tmDO, tmDQ, lse, delta, (__nv_bfloat16*)dqkv, S, H, scale, \
                                                                  causal ? 1 : 0, sched, g_dq_acc, dq_red, alibi_slopes); \
  }
  const int grid2 = 2 * sched.n_items < sms ? 2 * sched.n_items : sms;   // d_head 128: two passes per item
  if (dh == 64 && !alibi_slopes) PB_BWD(64, false, grid)
  else if (dh == 64) PB_BWD(64, true, grid)
  else if (!alibi_slopes) PB_BWD(128, false, grid2)
  else PB_BWD(128, true, grid2)
#undef PB_BWD
  attn_bwd_dq_convert_kernel<<<148 * 8, 256, 0, st>>>(g_dq_acc, (__nv_bfloat16*)dqkv, rows, d, scale);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) throw std::runtime_error(std::string("attention bwd launch: ") + cudaGetErrorString(e));
  return 3;
}

// ---------------------------------------------------------------------------------------------- RoPE
// In-place rotary embedding (rotate-half / GPT-NeoX convention) on the q and k thirds of a fused qkv buffer
// [T, 3*H*dh] bf16; cos / sin: fp32 [S, dh/2]. inverse = 1 applies the transposed rotation (gradients of q, k).
namespace {
__global__ void __launch_bounds__(256) rope_kernel(__nv_bfloat16* __restrict__ qkv, const float* __restrict__ cosT, const float* __restrict__ sinT,
                                                   long long T, int S, int H, int dh, int inverse) {
  const int half = dh / 2, groups = half / 8;                 // 8 pairs (16 bytes of each half) per thread
  const long long n = T * 2 * H * groups;                     // (token, q|k, head, group)
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int g = int(i % groups);
    long long r = i / groups;
    const int h = int(r % H);
    r /= H;
    const int which = int(r % 2);
    const long long t = r / 2;
    const int pos = int(t % S);
    __nv_bfloat16* base = qkv + t * (3LL * H * dh) + (long long)which * H * dh + h * dh + g * 8;
    uint4 a = *reinterpret_cast<const uint4*>(base);
    uint4 b = *reinterpret_cast<const uint4*>(base + half);
    rope_rotate8(a, b, cosT + (long long)pos * half + g * 8, sinT + (long long)pos * half + g * 8, inverse);
    *reinterpret_cast<uint4*>(base) = a;
    *reinterpret_cast<uint4*>(base + half) = b;
  }
}
}  // namespace

void rope_launch(void* qkv, const float* cosT, const float* sinT, long long T, int S, int H, int dh, bool inverse, cudaStream_t st) {
  if (dh % 16) throw std::runtime_error("photon_b200 rope: d_head must be a multiple of 16");
  const long long n = T * 2 * H * (dh / 16);
  const int blocks = int(std::min<long long>((n + 255) / 256, 148 * 16));
  rope_kernel<<<blocks, 256, 0, st>>>((__nv_bfloat16*)qkv, cosT, sinT, T, S, H, dh, inverse ? 1 : 0);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) throw std::runtime_error(std::string("rope launch: ") + cudaGetErrorString(e));
}

}  // namespace pb
