// rows.cuh -- the per-row maths of K2 and of the scatter half of K4, shared by gather.cu and xchg.cu:
//   F.normalize(p=2, dim=1, eps=1e-12) (V2.py:138) of one anchor row and its autograd backward.
// One warp holds one row.  Every kernel but k_gather_p2p gives lane l the channels l + 32 q (q < 8), so the NCHW and
// the channels-last kernels sum in the same order and their rows are equal bit for bit; keep it so.
#pragma once
#include "common.cuh"

namespace mscs {

constexpr int kMaxC = 256;      // channels of a row: 8 per lane

// the item of a batched launch that this block belongs to; block0: the items' first blocks, in ascending order
__device__ __forceinline__ int batch_item(const int* block0, int count) {
  int s = 0;
  while (s + 1 < count && (int)blockIdx.x >= block0[s + 1]) ++s;
  return s;
}

// 1 / max(||x||, 1e-12) of the row whose lane-held values are v: the lane's fmaf sum of squares in index order, then
// warp_sum.  Holds for any fixed assignment of 8 channels per lane.
__device__ __forceinline__ float inv_norm_of(const float (&v)[kMaxC / 32]) {
  float ss = 0.f;
#pragma unroll
  for (int q = 0; q < kMaxC / 32; ++q) ss = fmaf(v[q], v[q], ss);
  ss = warp_sum(ss);
  return 1.f / fmaxf(sqrtf(ss), 1e-12f);
}

// the unit row v * inv (lane l: channels l + 32 q): fp32 into f32_row[0, C), bf16 through put(c, value) for every
// c < C_pad, with zeros in [C, C_pad) (the similarity kernels read whole 64-channel blocks)
template <typename PutBf16>
__device__ __forceinline__ void store_unit_row(const float (&v)[kMaxC / 32], float inv, int C, int C_pad,
                                               float* f32_row, PutBf16 put) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int q = 0; q < kMaxC / 32; ++q) {
    const int c = lane + 32 * q;
    const float f = v[q] * inv;
    if (c < C) f32_row[c] = f;
    if (c < C_pad) put(c, __float2bfloat16(c < C ? f : 0.f));
  }
}
__device__ __forceinline__ void store_unit_row(const float (&v)[kMaxC / 32], float inv, int C, int C_pad,
                                               float* f32_row, __nv_bfloat16* bf16_row) {
  store_unit_row(v, inv, C, C_pad, f32_row, [bf16_row](int c, __nv_bfloat16 h) { bf16_row[c] = h; });
}

// Normalisation backward of row `row` (lane l: channels l + 32 q): dx = (g - f (f.g)) * inv from its gradient row g, its
// unit row f and inv = inv_norm[row].  Where ||x|| <= eps F.normalize divides by the constant eps, so there dx = g * inv.
// g may be the row dx is stored into afterwards (k_dx_rows): no __restrict__ here.
__device__ __forceinline__ void dx_row(const float* g, const float* f, const float* inv_norm, int row, int C,
                                       float (&dx)[kMaxC / 32]) {
  const int lane = threadIdx.x & 31;
  float gv[kMaxC / 32], fv[kMaxC / 32], dot = 0.f;
#pragma unroll
  for (int q = 0; q < kMaxC / 32; ++q) {
    const int c = lane + 32 * q;
    gv[q] = (c < C) ? g[c] : 0.f;
    fv[q] = (c < C) ? f[c] : 0.f;
    dot = fmaf(gv[q], fv[q], dot);
  }
  dot = warp_sum(dot);
  const float inv = inv_norm[row];
  const bool clamped = inv >= 1e12f;
#pragma unroll
  for (int q = 0; q < kMaxC / 32; ++q) dx[q] = (clamped ? gv[q] : (gv[q] - fv[q] * dot)) * inv;
}

}  // namespace mscs
