// Rotary embedding arithmetic shared by the training kernel (rope_kernel, attention_tcgen05.cu) and the decode-time
// KV-cache write (kv_write_kernel, decode.cu): both go through this one function, so a key rotated while decoding is
// bit-identical to the same key rotated by the training forward at the same position.
#pragma once
#include "ptx.cuh"

namespace pb {

// 8 rotate-half pairs: a = x[i..i+8), b = x[i+dh/2..i+dh/2+8) of one head; c / sn = cos / sin at (pos, i..i+8).
// inverse = 1 applies the transposed rotation.
__device__ __forceinline__ void rope_rotate8(uint4& a, uint4& b, const float* c, const float* sn, int inverse) {
  const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, bw[4] = {b.x, b.y, b.z, b.w};
  uint32_t oa[4], ob[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float2 x1 = unpack_bf16(aw[k]), x2 = unpack_bf16(bw[k]);
    const float c0 = c[2 * k], c1 = c[2 * k + 1];
    const float s0 = inverse ? -sn[2 * k] : sn[2 * k], s1 = inverse ? -sn[2 * k + 1] : sn[2 * k + 1];
    oa[k] = pack_bf16(x1.x * c0 - x2.x * s0, x1.y * c1 - x2.y * s1);
    ob[k] = pack_bf16(x2.x * c0 + x1.x * s0, x2.y * c1 + x1.y * s1);
  }
  a = make_uint4(oa[0], oa[1], oa[2], oa[3]);
  b = make_uint4(ob[0], ob[1], ob[2], ob[3]);
}

}  // namespace pb
