// Host API of the KV-cached decoding kernels (see decode.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace pb {

constexpr int DECODE_TILE_KEYS = 32;   // keys per shared-memory ring stage of decode_attention

// Number of key splits decode_attention uses for B*H (row, head) pairs over a cache of s_max positions: enough CTAs for
// about eight per SM (each CTA walks its tiles one after another), never more than one split per tile of keys. Fixed per
// (B, H, s_max), so a captured step stays valid.
int decode_attention_splits(int BH, int s_max, int num_sms);

// q: bf16 rows [B, ldq] (the q third of the step's qkv, RoPE applied); kv: bf16 [B, s_max, 2*H*dh] (k | v, head-major);
// lengths: int32 [B] valid keys per row (device); alibi: optional fp32 [H]; out: bf16 [B, H*dh]; lse: optional fp32 [B, H];
// scratch: fp32 [B*H*n_split*(dh+2)] when n_split > 1. Returns the number of kernels launched.
int decode_attention_launch(const void* q, long long ldq, const void* kv, int B, int s_max, int H, int dh, const int* lengths,
                            const float* alibi, float scale, int n_split, float* scratch, void* out, float* lse, cudaStream_t st);

// cache[b_idx[t], pos[t]] = k|v thirds of qkv row t; with rotate (cos / sin fp32 [>= s_max, dh/2]) q and k of the row are
// first rotated in place at pos[t], with the same arithmetic as rope_launch.
void kv_write_launch(void* qkv, long long ldq, void* cache, int B, int s_max, const int* b_idx, const int* pos, const float* cosT,
                     const float* sinT, long long T, int H, int dh, bool rotate, cudaStream_t st);

// out[r] = argmax_j logits[r, j] over bf16 rows [R, V] (row stride ld); ties go to the lowest index
void argmax_rows_launch(const void* logits, long long ld, long long R, int V, int64_t* out, cudaStream_t st);

}  // namespace pb
