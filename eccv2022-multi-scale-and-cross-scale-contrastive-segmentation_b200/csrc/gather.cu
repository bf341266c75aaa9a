// gather.cu -- K2 (gather sampled embeddings + L2 normalise) and the scatter half of K4
// (normalisation backward + dense gradient).
//   gather  : features[b,:,idx] (V2.py:123) + F.normalize(p=2, dim=1, eps=1e-12) (V2.py:138)
//   scatter : autograd backward of both: dx = (dF - f (f.dF)) / max(||x||, eps), written into
//             a dense zero (n,C,h,w) gradient at the sampled pixels.
// HBM-bound byte movers: NCHW means one anchor is C scalars `plane` floats apart (one 32 B
// sector per useful 4 B), so one warp owns one anchor and keeps 8 independent loads in flight.
#include "common.cuh"

namespace mscs {

constexpr int kMaxC = 256;

__global__ void __launch_bounds__(256)
k_gather_normalize(const float* __restrict__ feat, int C, int C_pad, int plane, const int* __restrict__ pix,
                   int N, int N_pad, __nv_bfloat16* __restrict__ anc_bf16, float* __restrict__ anc_f32,
                   float* __restrict__ inv_norm) {
  pdl_trigger();
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= N_pad) return;
  __nv_bfloat16* orow = anc_bf16 + (size_t)row * C_pad;
  if (row >= N) {                       // zero padding rows (TMA tiles read them)
    for (int c = lane; c < C_pad; c += 32) orow[c] = __float2bfloat16(0.f);
    return;
  }
  const int gp = pix[row];
  if (gp < 0) {                         // pooled mode: the row is owned by another rank (all-reduced later)
    for (int c = lane; c < C_pad; c += 32) orow[c] = __float2bfloat16(0.f);
    return;
  }
  const int b = gp / plane, p = gp - b * plane;
  const float* src = feat + ((size_t)b * C) * plane + p;
  float v[kMaxC / 32];
  float ss = 0.f;
#pragma unroll
  for (int j = 0; j < kMaxC / 32; ++j) {
    int c = lane + 32 * j;
    v[j] = (c < C) ? __ldg(src + (size_t)c * plane) : 0.f;
  }
#pragma unroll
  for (int j = 0; j < kMaxC / 32; ++j) ss = fmaf(v[j], v[j], ss);
  ss = warp_sum(ss);
  const float inv = 1.f / fmaxf(sqrtf(ss), 1e-12f);
  if (lane == 0) inv_norm[row] = inv;
#pragma unroll
  for (int j = 0; j < kMaxC / 32; ++j) {
    int c = lane + 32 * j;
    float f = v[j] * inv;
    if (c < C) anc_f32[(size_t)row * C + c] = f;
    if (c < C_pad) orow[c] = __float2bfloat16(c < C ? f : 0.f);
  }
}

__global__ void __launch_bounds__(256)
k_scatter_grad(const float* __restrict__ dF, int ldF, const float* __restrict__ anc_f32,
               const float* __restrict__ inv_norm, const int* __restrict__ pix, int N, int C, int plane,
               float* __restrict__ dfeat) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= N) return;
  const float* g = dF + (size_t)row * ldF;
  const float* f = anc_f32 + (size_t)row * C;
  float gv[kMaxC / 32], fv[kMaxC / 32];
  float dot = 0.f;
#pragma unroll
  for (int j = 0; j < kMaxC / 32; ++j) {
    int c = lane + 32 * j;
    gv[j] = (c < C) ? g[c] : 0.f;
    fv[j] = (c < C) ? f[c] : 0.f;
    dot = fmaf(gv[j], fv[j], dot);
  }
  dot = warp_sum(dot);
  const float inv = inv_norm[row];
  const bool clamped = inv >= 1e12f;        // ||x|| <= eps: F.normalize divides by the constant eps
  const int gp = pix[row];
  if (gp < 0) return;
  const int b = gp / plane, p = gp - b * plane;
  float* dst = dfeat + ((size_t)b * C) * plane + p;
#pragma unroll
  for (int j = 0; j < kMaxC / 32; ++j) {
    int c = lane + 32 * j;
    if (c < C) dst[(size_t)c * plane] = (clamped ? gv[j] : (gv[j] - fv[j] * dot)) * inv;
  }
}

// Gather in ADDRESS order: one warp per 8-pixel octet of the slot map (18% of them hold a sampled
// pixel at cfg-2).  Neighbouring warps then touch neighbouring 32-byte sectors of the same channel
// planes, so the 256 strided sector reads of an anchor hit open DRAM pages instead of random ones.
template <typename T>
__device__ __forceinline__ void
gather_sectors_body(int block, int nblocks, const T* __restrict__ feat, int C, int C_pad, int plane,
                    const int* __restrict__ slot, int n_octets, __nv_bfloat16* __restrict__ anc_bf16,
                    float* __restrict__ anc_f32, float* __restrict__ inv_norm, const int* __restrict__ n_rows_dev) {
  const int lane = threadIdx.x & 31;
  if (n_rows_dev != nullptr && block == nblocks - 1) {
    // device-driven call: the row count is only known on the device; this (extra) block zeroes the padding
    // rows [N, N_pad) of the operand matrix that the TMA tiles read
    const int N = *n_rows_dev, N_pad = (N + 255) / 256 * 256;
    uint32_t* z = reinterpret_cast<uint32_t*>(anc_bf16 + (size_t)N * C_pad);
    for (int i = threadIdx.x; i < (N_pad - N) * (C_pad / 2); i += blockDim.x) z[i] = 0u;
    return;
  }
  const int oct = block * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (oct >= n_octets) return;
  const int gp = oct * 8;
  const int s_mine = (lane < 8) ? slot[gp + lane] : -1;
  unsigned act = __ballot_sync(0xffffffffu, s_mine >= 0);
  if (act == 0) return;
  const int b = gp / plane, p = gp - b * plane;
  const T* src0 = feat + ((size_t)b * C) * plane + p;
  while (act) {
    const int j = __ffs(act) - 1;
    act &= act - 1;
    const int row = __shfl_sync(0xffffffffu, s_mine, j);
    const T* src = src0 + j;
    float v[kMaxC / 32];
    float ss = 0.f;
#pragma unroll
    for (int q = 0; q < kMaxC / 32; ++q) {
      const int c = lane + 32 * q;
      v[q] = (c < C) ? to_f32(__ldg(src + (size_t)c * plane)) : 0.f;
    }
#pragma unroll
    for (int q = 0; q < kMaxC / 32; ++q) ss = fmaf(v[q], v[q], ss);
    if (anc_bf16 == nullptr) {      // raw mode (projector-tail path): the sampled rows as they are, no normalisation
#pragma unroll
      for (int q = 0; q < kMaxC / 32; ++q) {
        const int c = lane + 32 * q;
        if (c < C) anc_f32[(size_t)row * C + c] = v[q];
      }
      continue;
    }
    ss = warp_sum(ss);
    const float inv = 1.f / fmaxf(sqrtf(ss), 1e-12f);
    if (lane == 0) inv_norm[row] = inv;
    __nv_bfloat16* orow = anc_bf16 + (size_t)row * C_pad;
#pragma unroll
    for (int q = 0; q < kMaxC / 32; ++q) {
      const int c = lane + 32 * q;
      const float f = v[q] * inv;
      if (c < C) anc_f32[(size_t)row * C + c] = f;
      if (c < C_pad) orow[c] = __float2bfloat16(c < C ? f : 0.f);
    }
  }
}

__global__ void __launch_bounds__(256)
k_gather_sectors(const float* __restrict__ feat, int C, int C_pad, int plane, const int* __restrict__ slot,
                 int n_octets, __nv_bfloat16* __restrict__ anc_bf16, float* __restrict__ anc_f32,
                 float* __restrict__ inv_norm, const int* __restrict__ n_rows_dev) {
  pdl_trigger();
  gather_sectors_body<float>(blockIdx.x, gridDim.x, feat, C, C_pad, plane, slot, n_octets, anc_bf16, anc_f32, inv_norm,
                      n_rows_dev);
}

// all scales of a call in ONE launch (the per-scale launches of the small scales do not fill the GPU and each
// costs a launch gap): block -> scale through the block prefix.  One instantiation per element type of the maps; a
// call that mixes types launches once per type present.
struct GatherBatch {
  const void* feat[MSCS_MAX_SCALES]; const int* slot[MSCS_MAX_SCALES]; const int* n_rows_dev[MSCS_MAX_SCALES];
  __nv_bfloat16* bf16[MSCS_MAX_SCALES]; float* f32[MSCS_MAX_SCALES]; float* inv[MSCS_MAX_SCALES];
  int C[MSCS_MAX_SCALES], plane[MSCS_MAX_SCALES], n_oct[MSCS_MAX_SCALES], block0[MSCS_MAX_SCALES + 1];
  int count;
};
template <typename T>
__global__ void __launch_bounds__(256) k_gather_sectors_batch(const __grid_constant__ GatherBatch g) {
  pdl_trigger();      // the next kernel of the forward (k_row_ranges) is launched programmatically, see common.cuh
  int s = 0;
  while (s + 1 < g.count && (int)blockIdx.x >= g.block0[s + 1]) ++s;
  gather_sectors_body<T>(blockIdx.x - g.block0[s], g.block0[s + 1] - g.block0[s], static_cast<const T*>(g.feat[s]), g.C[s],
                      (g.C[s] + 63) / 64 * 64, g.plane[s], g.slot[s], g.n_oct[s], g.bf16[s], g.f32[s], g.inv[s],
                      g.n_rows_dev[s]);
}

// Projector-tail path: the sampled c-vectors as they are (no normalisation), same octet walk.  The slot map holds the
// sampled rows only, so the row count is not needed; rows the call does not sample are not touched.
template <typename T>
__global__ void __launch_bounds__(256) k_gather_raw_batch(const __grid_constant__ GatherBatch g) {
  int s = 0;
  while (s + 1 < g.count && (int)blockIdx.x >= g.block0[s + 1]) ++s;
  gather_sectors_body<T>(blockIdx.x - g.block0[s], g.block0[s + 1] - g.block0[s], static_cast<const T*>(g.feat[s]), g.C[s],
                         0, g.plane[s], g.slot[s], g.n_oct[s], nullptr, g.f32[s], nullptr, nullptr);
}

// slot map: slot[image*plane + pixel] = sorted anchor row sampled there, or -1
__global__ void k_slot_map(const int* __restrict__ pix, int N, int* __restrict__ slot) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N && pix[i] >= 0) slot[pix[i]] = i;      // negative: row owned by another rank (pooled mode)
}

// Sector writer: the dense gradient is already zero; one warp per 8-pixel octet (= one 32-byte
// sector per channel plane) rewrites every sector that holds at least one sampled pixel with
// full-sector stores (values + explicit zeros), so no partial-sector read-modify-write reaches HBM.
// pooled mode: gradient row i was computed by rank i / rows_per_rank and is READ FROM THAT RANK'S slab over NVLink
// (n == 0: every row is local, `dF` is used)
struct PullRows { const float* p[MSCS_MAX_RANKS]; int n, rows_per_rank; };

__device__ __forceinline__ void
scatter_sectors_body(const float* __restrict__ dF, int ldF, const float* __restrict__ anc_f32,
                  const float* __restrict__ inv_norm, const int* __restrict__ slot, int n_octets, int C,
                  int plane, float* __restrict__ dfeat, int block_base, const PullRows* pull = nullptr) {
  const int lane = threadIdx.x & 31;
  const int oct = ((int)blockIdx.x - block_base) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (oct >= n_octets) return;
  const int gp = oct * 8;
  const int s_mine = (lane < 8) ? slot[gp + lane] : -1;
  if (__ballot_sync(0xffffffffu, s_mine >= 0) == 0) return;
  const int b = gp / plane, p = gp - b * plane;
  float dx[8][kMaxC / 32];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int row = __shfl_sync(0xffffffffu, s_mine, j);
    if (row >= 0) {                                   // warp-uniform
      const float* g = (pull ? pull->p[row / pull->rows_per_rank] : dF) + (size_t)row * ldF;
      const float* f = anc_f32 + (size_t)row * C;
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
      for (int q = 0; q < kMaxC / 32; ++q) dx[j][q] = (clamped ? gv[q] : (gv[q] - fv[q] * dot)) * inv;
    } else {
#pragma unroll
      for (int q = 0; q < kMaxC / 32; ++q) dx[j][q] = 0.f;
    }
  }
#pragma unroll
  for (int q = 0; q < kMaxC / 32; ++q) {
    const int c = lane + 32 * q;
    if (c < C) {
      float4* dst = reinterpret_cast<float4*>(dfeat + ((size_t)b * C + c) * plane + p);
      dst[0] = make_float4(dx[0][q], dx[1][q], dx[2][q], dx[3][q]);
      dst[1] = make_float4(dx[4][q], dx[5][q], dx[6][q], dx[7][q]);
    }
  }
}

__global__ void __launch_bounds__(256)
k_scatter_sectors_pull(const __grid_constant__ PullRows pull, int ldF, const float* __restrict__ anc_f32,
                       const float* __restrict__ inv_norm, const int* __restrict__ slot, int n_octets, int C,
                       int plane, float* __restrict__ dfeat) {
  scatter_sectors_body(nullptr, ldF, anc_f32, inv_norm, slot, n_octets, C, plane, dfeat, 0, &pull);
}


// ---------------------------------------------------------------------------------------
// Dense gradient in ONE streaming pass: every byte of the dense gradient is written exactly once, zeros and values
// alike, so no zero fill has to run ahead of the backward (a 535 MB fill at cfg-2 is not hidden by overlapping it:
// memset / copy kernels take the SMs away from whatever they run next to, ~70 us of step time wherever it was put).
//   k_dx_rows:      dF row -> dx row in place   (normalisation backward, N x C, tiny)
//   k_dense_stream: out[b][c][p..p+P) = slot[b][p+i] >= 0 ? dx[slot][c] : 0   (below, after the channels-last kernels)
// ---------------------------------------------------------------------------------------
struct DenseBatch {
  float* dF[MSCS_MAX_SCALES]; const float* f32[MSCS_MAX_SCALES]; const float* inv[MSCS_MAX_SCALES];
  const int* slot[MSCS_MAX_SCALES]; const int* n_rows_dev[MSCS_MAX_SCALES];
  int ldF[MSCS_MAX_SCALES], C[MSCS_MAX_SCALES], plane[MSCS_MAX_SCALES], n[MSCS_MAX_SCALES], rows[MSCS_MAX_SCALES];
  int rowblk0[MSCS_MAX_SCALES + 1];         // block prefix of the row kernel (8 rows per block)
  int count;
};

__global__ void __launch_bounds__(256) k_dx_rows(const __grid_constant__ DenseBatch g) {
  int s = 0;
  while (s + 1 < g.count && (int)blockIdx.x >= g.rowblk0[s + 1]) ++s;
  const int lane = threadIdx.x & 31;
  const int row = ((int)blockIdx.x - g.rowblk0[s]) * 8 + (threadIdx.x >> 5);
  // rows[s] sizes the grid; with a device-resident count it is an upper bound and the rows beyond the count are stale
  if (row >= g.rows[s] || (g.n_rows_dev[s] && row >= *g.n_rows_dev[s])) return;
  const int C = g.C[s];
  float* gr = g.dF[s] + (size_t)row * g.ldF[s];
  const float* f = g.f32[s] + (size_t)row * C;
  float gv[kMaxC / 32], fv[kMaxC / 32], dot = 0.f;
#pragma unroll
  for (int q = 0; q < kMaxC / 32; ++q) {
    const int c = lane + 32 * q;
    gv[q] = (c < C) ? gr[c] : 0.f;
    fv[q] = (c < C) ? f[c] : 0.f;
    dot = fmaf(gv[q], fv[q], dot);
  }
  dot = warp_sum(dot);
  const float inv = g.inv[s][row];
  const bool clamped = inv >= 1e12f;        // ||x|| <= eps: F.normalize divides by the constant eps
#pragma unroll
  for (int q = 0; q < kMaxC / 32; ++q) {
    const int c = lane + 32 * q;
    if (c < C) gr[c] = (clamped ? gv[q] : (gv[q] - fv[q] * dot)) * inv;
  }
}


// ---------------------------------------------------------------------------------------
// Channels-last feature maps (memory order [n][h][w][C], e.g. a projector run in torch.channels_last): an anchor is
// ONE contiguous row of C floats instead of C sectors `plane` floats apart, so gather and scatter become plain row
// copies (33 MB instead of 354 MB of DRAM reads at cfg-2).  Warp per sorted anchor row; lane l handles the channels
// l + 32 q -- the same lane/channel assignment as the NCHW kernels, so the results are bit-identical.
// ---------------------------------------------------------------------------------------
struct RowsBatch {
  const void* feat[MSCS_MAX_SCALES]; const int* pix[MSCS_MAX_SCALES]; const int* n_rows_dev[MSCS_MAX_SCALES];
  __nv_bfloat16* bf16[MSCS_MAX_SCALES]; float* f32[MSCS_MAX_SCALES]; float* inv[MSCS_MAX_SCALES];
  const float* dF[MSCS_MAX_SCALES]; void* dfeat[MSCS_MAX_SCALES];
  int C[MSCS_MAX_SCALES], ldF[MSCS_MAX_SCALES], rows[MSCS_MAX_SCALES], block0[MSCS_MAX_SCALES + 1];
  int count;
};

template <typename T>
__global__ void __launch_bounds__(256) k_gather_rows_nhwc(const __grid_constant__ RowsBatch g) {
  pdl_trigger();
  int s = 0;
  while (s + 1 < g.count && (int)blockIdx.x >= g.block0[s + 1]) ++s;
  const int lane = threadIdx.x & 31;
  const int row = ((int)blockIdx.x - g.block0[s]) * 8 + (threadIdx.x >> 5);
  const int N = g.n_rows_dev[s] ? *g.n_rows_dev[s] : g.rows[s], N_pad = (N + 255) / 256 * 256;
  if (row >= N_pad) return;
  const int C = g.C[s], C_pad = (C + 63) / 64 * 64;
  __nv_bfloat16* orow = g.bf16[s] + (size_t)row * C_pad;
  const int gp = row < N ? g.pix[s][row] : -1;
  if (gp < 0) {                         // padding row, or (pooled mode) a row owned by another rank
    for (int c = lane; c < C_pad; c += 32) orow[c] = __float2bfloat16(0.f);
    return;
  }
  const T* src = static_cast<const T*>(g.feat[s]) + (size_t)gp * C;
  float v[kMaxC / 32];
  float ss = 0.f;
#pragma unroll
  for (int q = 0; q < kMaxC / 32; ++q) {
    const int c = lane + 32 * q;
    v[q] = (c < C) ? to_f32(__ldg(src + c)) : 0.f;
  }
#pragma unroll
  for (int q = 0; q < kMaxC / 32; ++q) ss = fmaf(v[q], v[q], ss);
  ss = warp_sum(ss);
  const float inv = 1.f / fmaxf(sqrtf(ss), 1e-12f);
  if (lane == 0) g.inv[s][row] = inv;
#pragma unroll
  for (int q = 0; q < kMaxC / 32; ++q) {
    const int c = lane + 32 * q;
    const float f = v[q] * inv;
    if (c < C) g.f32[s][(size_t)row * C + c] = f;
    if (c < C_pad) orow[c] = __float2bfloat16(c < C ? f : 0.f);
  }
}

// normalisation backward + row store into the (pre-zeroed) channels-last dense gradient
template <typename T>
__global__ void __launch_bounds__(256) k_scatter_rows_nhwc(const __grid_constant__ RowsBatch g) {
  int s = 0;
  while (s + 1 < g.count && (int)blockIdx.x >= g.block0[s + 1]) ++s;
  const int lane = threadIdx.x & 31;
  const int row = ((int)blockIdx.x - g.block0[s]) * 8 + (threadIdx.x >> 5);
  if (row >= g.rows[s] || (g.n_rows_dev[s] && row >= *g.n_rows_dev[s])) return;      // (as k_dx_rows)
  const int gp = g.pix[s][row];
  if (gp < 0) return;
  const int C = g.C[s];
  const float* gr = g.dF[s] + (size_t)row * g.ldF[s];
  const float* f = g.f32[s] + (size_t)row * C;
  float gv[kMaxC / 32], fv[kMaxC / 32], dot = 0.f;
#pragma unroll
  for (int q = 0; q < kMaxC / 32; ++q) {
    const int c = lane + 32 * q;
    gv[q] = (c < C) ? gr[c] : 0.f;
    fv[q] = (c < C) ? f[c] : 0.f;
    dot = fmaf(gv[q], fv[q], dot);
  }
  dot = warp_sum(dot);
  const float inv = g.inv[s][row];
  const bool clamped = inv >= 1e12f;        // ||x|| <= eps: F.normalize divides by the constant eps
  T* dst = static_cast<T*>(g.dfeat[s]) + (size_t)gp * C;
#pragma unroll
  for (int q = 0; q < kMaxC / 32; ++q) {
    const int c = lane + 32 * q;
    if (c < C) dst[c] = from_f32<T>((clamped ? gv[q] : (gv[q] - fv[q] * dot)) * inv);
  }
}

// Projector-tail path, channels-last: raw row copies in both directions (warp per sorted row, rows below the count)
//   gather: rows[row][:] = feat[pix[row]][:]  (fp32 rows)      store: dfeat[pix[row]][:] = rows[row][:]  (map's type)
template <typename T, bool GATHER>
__global__ void __launch_bounds__(256) k_rows_raw_nhwc(const __grid_constant__ RowsBatch g) {
  int s = 0;
  while (s + 1 < g.count && (int)blockIdx.x >= g.block0[s + 1]) ++s;
  const int lane = threadIdx.x & 31;
  const int row = ((int)blockIdx.x - g.block0[s]) * 8 + (threadIdx.x >> 5);
  if (row >= g.rows[s] || (g.n_rows_dev[s] && row >= *g.n_rows_dev[s])) return;
  const int gp = g.pix[s][row];
  if (gp < 0) return;
  const int C = g.C[s];
  if (GATHER) {
    const T* src = static_cast<const T*>(g.feat[s]) + (size_t)gp * C;
    float* dst = g.f32[s] + (size_t)row * C;
    for (int c = lane; c < C; c += 32) dst[c] = to_f32(__ldg(src + c));
  } else {
    const float* src = g.dF[s] + (size_t)row * g.ldF[s];
    T* dst = static_cast<T*>(g.dfeat[s]) + (size_t)gp * C;
    for (int c = lane; c < C; c += 32) dst[c] = from_f32<T>(src[c]);
  }
}

// One-pass dense writer: a thread OWNS 4 consecutive pixels and walks the channel planes.
// Its four slot entries are fetched once (one coalesced int4), so the sampled / not-sampled decision is loop
// invariant: 97 % of the threads run a pure store loop, the others add up to four independent (predicated) loads of
// dx[row][c] per channel.  A block writes 2 KB contiguous per channel plane (512 pixels), i.e. whole DRAM pages in
// linear order per plane -- the order of the memset it replaces, without its second pass over the sampled sectors.
// Half gradients: a thread owns 8 pixels (two int4 of slot entries, up to eight loads per channel) so that every store
// is still 16 bytes; a block then covers 1024 pixels.  (The fast path guarantees planes that are a multiple of 8.)
struct DenseStream {
  const float* dx[MSCS_MAX_SCALES]; const int* slot[MSCS_MAX_SCALES]; void* dfeat[MSCS_MAX_SCALES];
  int ld[MSCS_MAX_SCALES], C[MSCS_MAX_SCALES], plane[MSCS_MAX_SCALES], npix[MSCS_MAX_SCALES], blk0[MSCS_MAX_SCALES + 1];
  int count;
};
template <typename T>
__global__ void __launch_bounds__(128) k_dense_stream(const __grid_constant__ DenseStream g) {
  constexpr int P = 16 / sizeof(T);      // pixels per thread: one 16-byte store per channel plane
  int s = 0;
  while (s + 1 < g.count && (int)blockIdx.x >= g.blk0[s + 1]) ++s;
  const int lin = (((int)blockIdx.x - g.blk0[s]) * 128 + (int)threadIdx.x) * P;
  if (lin >= g.npix[s]) return;
  const int plane = g.plane[s], C = g.C[s], ld = g.ld[s];
  int sl[P];
#pragma unroll
  for (int i = 0; i < P; i += 4) {
    const int4 q = *reinterpret_cast<const int4*>(g.slot[s] + lin + i);
    sl[i] = q.x; sl[i + 1] = q.y; sl[i + 2] = q.z; sl[i + 3] = q.w;
  }
  const int b = lin / plane, p = lin - b * plane;
  T* __restrict__ out = static_cast<T*>(g.dfeat[s]) + ((size_t)b * C) * plane + p;
  const float* __restrict__ dx = g.dx[s];
  const float* r[P];
  bool h[P];
#pragma unroll
  for (int i = 0; i < P; ++i) { r[i] = dx + (size_t)max(sl[i], 0) * ld; h[i] = sl[i] >= 0; }
#pragma unroll 8
  for (int c = 0; c < C; ++c) {
    float v[P];
#pragma unroll
    for (int i = 0; i < P; ++i) v[i] = h[i] ? __ldg(r[i] + c) : 0.f;
    st16_cs(out + (size_t)c * plane, v);
  }
}

}  // namespace mscs

using namespace mscs;

extern "C" int mscs_gather_normalize_sectors(const float* feat, int n, int C, int plane, const int32_t* slot, int N,
                                             void* anc_bf16, float* anc_f32, float* inv_norm, void* stream_) {
  MSCS_CHECK_ARG(feat && slot && anc_bf16 && anc_f32 && inv_norm, "null pointer argument");
  MSCS_CHECK_ARG(C >= 1 && C <= kMaxC, "C=%d unsupported (1..%d)", C, kMaxC);
  MSCS_CHECK_ARG(n >= 1 && plane >= 8 && plane % 8 == 0 && N >= 1, "bad sizes (plane must be a multiple of 8)");
  cudaStream_t st = (cudaStream_t)stream_;
  const int C_pad = (C + 63) / 64 * 64, N_pad = (N + 255) / 256 * 256;
  if (N_pad > N)      // zero padding rows of the operand matrix (TMA tiles read them)
    MSCS_CUDA(cudaMemsetAsync((__nv_bfloat16*)anc_bf16 + (size_t)N * C_pad, 0,
                              sizeof(__nv_bfloat16) * (size_t)(N_pad - N) * C_pad, st));
  const int n_oct = n * (plane / 8);
  k_gather_sectors<<<ceil_div(n_oct, 8), 256, 0, st>>>(feat, C, C_pad, plane, slot, n_oct, (__nv_bfloat16*)anc_bf16,
                                                       anc_f32, inv_norm, nullptr);
  MSCS_LAUNCH_CHECK();
  return 0;
}

extern "C" int mscs_slot_map(const int32_t* pix, int N, int n_pixels, int32_t* slot, void* stream_) {
  MSCS_CHECK_ARG(pix && slot && N >= 1 && n_pixels >= 1, "bad arguments");
  cudaStream_t st = (cudaStream_t)stream_;
  MSCS_CUDA(cudaMemsetAsync(slot, 0xff, sizeof(int) * (size_t)n_pixels, st));
  k_slot_map<<<ceil_div(N, 256), 256, 0, st>>>(pix, N, slot);
  MSCS_LAUNCH_CHECK();
  return 0;
}

// pooled mode: the same scatter with every gradient row read from the rank that computed it (row / rows_per_rank)
extern "C" int mscs_scatter_sectors_pull(void* const* slabs, int world, size_t dF_byte_off, int rows_per_rank, int ldF,
                                         const float* anc_f32, const float* inv_norm, const int32_t* slot, int n, int C,
                                         int plane, float* dfeat, void* stream_) {
  MSCS_CHECK_ARG(slabs && anc_f32 && inv_norm && slot && dfeat, "null pointer argument");
  MSCS_CHECK_ARG(world >= 1 && world <= MSCS_MAX_RANKS && rows_per_rank >= 1, "bad world %d / rows per rank %d", world,
                 rows_per_rank);
  MSCS_CHECK_ARG(C >= 1 && C <= kMaxC && ldF >= C, "C=%d / ldF=%d unsupported", C, ldF);
  MSCS_CHECK_ARG(plane % 8 == 0, "plane %d is not a multiple of 8 pixels", plane);
  PullRows pull{};
  pull.n = world; pull.rows_per_rank = rows_per_rank;
  for (int r = 0; r < world; ++r) {
    MSCS_CHECK_ARG(slabs[r] != nullptr, "peer %d: null slab pointer", r);
    pull.p[r] = reinterpret_cast<const float*>((const char*)slabs[r] + dF_byte_off);
  }
  const int n_oct = n * (plane / 8);
  k_scatter_sectors_pull<<<ceil_div(n_oct, 8), 256, 0, (cudaStream_t)stream_>>>(pull, ldF, anc_f32, inv_norm, slot,
                                                                                n_oct, C, plane, dfeat);
  MSCS_LAUNCH_CHECK();
  return 0;
}

// element-type checks shared by the batched entry points: a known MSCS_DTYPE_* code and an address aligned to `align`
// bytes (at least the element size)
static int check_dtype(int s, int dtype, const void* p, int align, const char* what) {
  MSCS_CHECK_ARG(dtype_bytes(dtype) > 0, "item %d: dtype %d unknown (MSCS_DTYPE_F32 / _BF16 / _F16)", s, dtype);
  const int a = align > dtype_bytes(dtype) ? align : dtype_bytes(dtype);
  MSCS_CHECK_ARG((uintptr_t)p % a == 0, "item %d: %s must be %d-byte aligned", s, what, a);
  return 0;
}

// the items of one element type, one launch
template <typename T>
static int gather_sectors_launch(const mscs_gather_item* items, int count, int dtype, cudaStream_t st, bool raw = false) {
  GatherBatch g{};
  int blocks = 0;
  for (int s = 0; s < count; ++s) {
    const mscs_gather_item& it = items[s];
    if (it.dtype != dtype) continue;
    const int j = g.count++;
    g.feat[j] = it.feat; g.slot[j] = it.slot; g.n_rows_dev[j] = it.n_rows_dev;
    g.bf16[j] = (__nv_bfloat16*)it.anc_bf16; g.f32[j] = it.anc_f32; g.inv[j] = it.inv_norm;
    g.C[j] = it.C; g.plane[j] = it.plane; g.n_oct[j] = it.n * (it.plane / 8);
  }
  if (g.count == 0) return 0;
  for (int j = 0; j < g.count; ++j) {
    g.block0[j] = blocks;
    blocks += ceil_div(g.n_oct[j], 8) + (raw ? 0 : 1);      // + the block that zeroes the padding rows
  }
  g.block0[g.count] = blocks;
  if (raw) k_gather_raw_batch<T><<<blocks, 256, 0, st>>>(g);
  else k_gather_sectors_batch<T><<<blocks, 256, 0, st>>>(g);
  MSCS_LAUNCH_CHECK();
  return 0;
}

// One launch for every scale of a call (see mscs.h)
extern "C" int mscs_gather_normalize_sectors_batch(const mscs_gather_item* items, int count, void* stream_) {
  MSCS_CHECK_ARG(items && count >= 1 && count <= MSCS_MAX_SCALES, "bad item count %d", count);
  for (int s = 0; s < count; ++s) {
    const mscs_gather_item& it = items[s];
    MSCS_CHECK_ARG(it.feat && it.slot && it.n_rows_dev && it.anc_bf16 && it.anc_f32 && it.inv_norm,
                   "item %d: null pointer argument", s);
    MSCS_CHECK_ARG(it.C >= 1 && it.C <= kMaxC, "item %d: C=%d unsupported (1..%d)", s, it.C, kMaxC);
    MSCS_CHECK_ARG(it.n >= 1 && it.plane >= 8 && it.plane % 8 == 0, "item %d: plane must be a multiple of 8", s);
    if (int rc = check_dtype(s, it.dtype, it.feat, 1, "feat")) return rc;
  }
  cudaStream_t st = (cudaStream_t)stream_;
  if (int rc = gather_sectors_launch<float>(items, count, MSCS_DTYPE_F32, st)) return rc;
  if (int rc = gather_sectors_launch<__nv_bfloat16>(items, count, MSCS_DTYPE_BF16, st)) return rc;
  return gather_sectors_launch<__half>(items, count, MSCS_DTYPE_F16, st);
}

// Projector-tail path: the raw rows of every scale, one launch per element type (see mscs.h)
extern "C" int mscs_gather_raw_batch(const mscs_gather_item* items, int count, void* stream_) {
  MSCS_CHECK_ARG(items && count >= 1 && count <= MSCS_MAX_SCALES, "bad item count %d", count);
  for (int s = 0; s < count; ++s) {
    const mscs_gather_item& it = items[s];
    MSCS_CHECK_ARG(it.feat && it.slot && it.anc_f32, "item %d: null pointer argument", s);
    MSCS_CHECK_ARG(it.C >= 1 && it.C <= kMaxC, "item %d: C=%d unsupported (1..%d)", s, it.C, kMaxC);
    MSCS_CHECK_ARG(it.n >= 1 && it.plane >= 8 && it.plane % 8 == 0, "item %d: plane must be a multiple of 8", s);
    if (int rc = check_dtype(s, it.dtype, it.feat, 1, "feat")) return rc;
  }
  cudaStream_t st = (cudaStream_t)stream_;
  if (int rc = gather_sectors_launch<float>(items, count, MSCS_DTYPE_F32, st, true)) return rc;
  if (int rc = gather_sectors_launch<__nv_bfloat16>(items, count, MSCS_DTYPE_BF16, st, true)) return rc;
  return gather_sectors_launch<__half>(items, count, MSCS_DTYPE_F16, st, true);
}

struct ScatterBatch {
  const float* dF[MSCS_MAX_SCALES]; const float* f32[MSCS_MAX_SCALES]; const float* inv[MSCS_MAX_SCALES];
  const int* slot[MSCS_MAX_SCALES]; float* dfeat[MSCS_MAX_SCALES];
  int ldF[MSCS_MAX_SCALES], C[MSCS_MAX_SCALES], plane[MSCS_MAX_SCALES], n_oct[MSCS_MAX_SCALES], block0[MSCS_MAX_SCALES + 1];
  int count;
};
__global__ void __launch_bounds__(256) k_scatter_sectors_batch(const __grid_constant__ ScatterBatch g) {
  int s = 0;
  while (s + 1 < g.count && (int)blockIdx.x >= g.block0[s + 1]) ++s;
  scatter_sectors_body(g.dF[s], g.ldF[s], g.f32[s], g.inv[s], g.slot[s], g.n_oct[s], g.C[s], g.plane[s], g.dfeat[s],
                       g.block0[s]);
}

extern "C" int mscs_scatter_sectors_batch(const mscs_scatter_item* items, int count, void* stream_) {
  MSCS_CHECK_ARG(items && count >= 1 && count <= MSCS_MAX_SCALES, "bad item count %d", count);
  ScatterBatch g{};
  g.count = count;
  int blocks = 0;
  for (int s = 0; s < count; ++s) {
    const mscs_scatter_item& it = items[s];
    MSCS_CHECK_ARG(it.dF && it.anc_f32 && it.inv_norm && it.slot && it.dfeat, "item %d: null pointer argument", s);
    MSCS_CHECK_ARG(it.C >= 1 && it.C <= kMaxC && it.ldF >= it.C, "item %d: C=%d / ldF=%d unsupported", s, it.C, it.ldF);
    MSCS_CHECK_ARG(it.plane % 8 == 0, "item %d: plane %d is not a multiple of 8 pixels", s, it.plane);
    if (int rc = check_dtype(s, it.dtype, it.dfeat, 16, "dfeat")) return rc;
    MSCS_CHECK_ARG(it.dtype == MSCS_DTYPE_F32, "item %d: the sector scatter writes fp32 gradients only", s);
    g.dF[s] = it.dF; g.f32[s] = it.anc_f32; g.inv[s] = it.inv_norm; g.slot[s] = it.slot; g.dfeat[s] = (float*)it.dfeat;
    g.ldF[s] = it.ldF; g.C[s] = it.C; g.plane[s] = it.plane; g.n_oct[s] = it.n * (it.plane / 8);
    g.block0[s] = blocks;
    blocks += ceil_div(g.n_oct[s], 8);
  }
  g.block0[count] = blocks;
  k_scatter_sectors_batch<<<blocks, 256, 0, (cudaStream_t)stream_>>>(g);
  MSCS_LAUNCH_CHECK();
  return 0;
}


extern "C" int mscs_gather_normalize(const float* feat, int n, int C, int plane, const int32_t* pix, int N,
                                     void* anc_bf16, float* anc_f32, float* inv_norm, void* stream_) {
  MSCS_CHECK_ARG(feat && pix && anc_bf16 && anc_f32 && inv_norm, "null pointer argument");
  MSCS_CHECK_ARG(C >= 1 && C <= kMaxC, "C=%d unsupported (1..%d)", C, kMaxC);
  MSCS_CHECK_ARG(n >= 1 && plane >= 1 && N >= 1, "bad sizes");
  const int C_pad = (C + 63) / 64 * 64, N_pad = (N + 255) / 256 * 256;
  k_gather_normalize<<<ceil_div(N_pad, 8), 256, 0, (cudaStream_t)stream_>>>(
      feat, C, C_pad, plane, pix, N, N_pad, (__nv_bfloat16*)anc_bf16, anc_f32, inv_norm);
  MSCS_LAUNCH_CHECK();
  return 0;
}

extern "C" int mscs_scatter_grad(const float* dF, int ldF, const float* anc_f32, const float* inv_norm,
                                 const int32_t* pix, int N, int n, int C, int plane, float* dfeat,
                                 int zero_fill, void* stream_) {
  MSCS_CHECK_ARG(dF && anc_f32 && inv_norm && pix && dfeat, "null pointer argument");
  MSCS_CHECK_ARG(C >= 1 && C <= kMaxC && ldF >= C, "C=%d / ldF=%d unsupported", C, ldF);
  cudaStream_t st = (cudaStream_t)stream_;
  if (zero_fill) MSCS_CUDA(cudaMemsetAsync(dfeat, 0, sizeof(float) * (size_t)n * C * plane, st));
  k_scatter_grad<<<ceil_div(N, 8), 256, 0, st>>>(dF, ldF, anc_f32, inv_norm, pix, N, C, plane, dfeat);
  MSCS_LAUNCH_CHECK();
  return 0;
}

// the dense writer over the items of one element type (128 threads x 16 / sizeof(T) pixels per block)
template <typename T>
static int dense_stream_launch(const DenseBatch& g, const mscs_scatter_item* items, int dtype, cudaStream_t st) {
  DenseStream d{};
  int blk = 0;
  for (int s = 0; s < g.count; ++s) {
    if (items[s].dtype != dtype) continue;
    const int j = d.count++;
    d.dx[j] = g.dF[s]; d.slot[j] = g.slot[s]; d.dfeat[j] = items[s].dfeat; d.ld[j] = g.ldF[s]; d.C[j] = g.C[s];
    d.plane[j] = g.plane[s]; d.npix[j] = g.n[s] * g.plane[s]; d.blk0[j] = blk;
    blk += ceil_div(d.npix[j], 128 * (16 / (int)sizeof(T)));
  }
  if (d.count == 0) return 0;
  d.blk0[d.count] = blk;
  k_dense_stream<T><<<blk, 128, 0, st>>>(d);
  MSCS_LAUNCH_CHECK();
  return 0;
}

extern "C" int mscs_scatter_dense_batch(const mscs_scatter_item* items, const int32_t* rows, int count, void* stream_) {
  MSCS_CHECK_ARG(items && rows && count >= 1 && count <= MSCS_MAX_SCALES, "bad arguments");
  DenseBatch g{};
  g.count = count;
  int rb = 0, n_raw = 0;
  for (int s = 0; s < count; ++s) {
    const mscs_scatter_item& it = items[s];
    MSCS_CHECK_ARG(it.dF && it.slot && it.dfeat, "item %d: null pointer argument", s);
    MSCS_CHECK_ARG((it.anc_f32 == nullptr) == (it.inv_norm == nullptr),
                   "item %d: anc_f32 and inv_norm must both be set or both be NULL (raw rows)", s);
    const bool raw = it.anc_f32 == nullptr;
    n_raw += raw;
    MSCS_CHECK_ARG(it.C >= 1 && it.C <= kMaxC && it.ldF >= it.C, "item %d: C=%d / ldF=%d unsupported", s, it.C, it.ldF);
    MSCS_CHECK_ARG(it.plane % 4 == 0 && rows[s] >= 0, "item %d: plane %d is not a multiple of 4 pixels", s, it.plane);
    if (int rc = check_dtype(s, it.dtype, it.dfeat, 16, "dfeat")) return rc;
    MSCS_CHECK_ARG(it.dtype == MSCS_DTYPE_F32 || it.plane % 8 == 0,
                   "item %d: half gradients need a plane that is a multiple of 8 pixels (plane %d)", s, it.plane);
    g.dF[s] = const_cast<float*>(it.dF); g.f32[s] = it.anc_f32; g.inv[s] = it.inv_norm; g.slot[s] = it.slot;
    g.ldF[s] = it.ldF; g.C[s] = it.C; g.plane[s] = it.plane; g.n[s] = it.n; g.rows[s] = raw ? 0 : rows[s];
    g.n_rows_dev[s] = it.n_rows_dev;
    MSCS_CHECK_ARG((long long)it.n * it.C * it.plane < (1ll << 32), "item %d: more than 2^32 gradient elements", s);
    g.rowblk0[s] = rb; rb += ceil_div(g.rows[s], 8);      // raw rows are written as they are: no blocks
  }
  g.rowblk0[count] = rb;
  cudaStream_t st = (cudaStream_t)stream_;
  if (n_raw < count) {
    k_dx_rows<<<rb > 0 ? rb : 1, 256, 0, st>>>(g);
    MSCS_LAUNCH_CHECK();
  }
  if (int rc = dense_stream_launch<float>(g, items, MSCS_DTYPE_F32, st)) return rc;
  if (int rc = dense_stream_launch<__nv_bfloat16>(g, items, MSCS_DTYPE_BF16, st)) return rc;
  return dense_stream_launch<__half>(g, items, MSCS_DTYPE_F16, st);
}

// ---- channels-last (NHWC) row gather / scatter, every scale of one element type in one launch (see mscs.h) ----
enum RowsKind { kRowsGather, kRowsScatter, kRowsGatherRaw };

static int rows_check(const mscs_rows_item* items, int count, RowsKind kind) {
  MSCS_CHECK_ARG(items && count >= 1 && count <= MSCS_MAX_SCALES, "bad item count %d", count);
  const bool gather = kind != kRowsScatter;
  for (int s = 0; s < count; ++s) {
    const mscs_rows_item& it = items[s];
    if (kind == kRowsScatter) {     // anc_f32 and inv_norm both NULL: the rows dF are stored as they are
      MSCS_CHECK_ARG(it.pix, "item %d: null pointer argument", s);
      MSCS_CHECK_ARG((it.anc_f32 == nullptr) == (it.inv_norm == nullptr),
                     "item %d: anc_f32 and inv_norm must both be set or both be NULL (raw rows)", s);
    } else {
      MSCS_CHECK_ARG(it.pix && it.anc_f32 && (kind == kRowsGatherRaw || it.inv_norm), "item %d: null pointer argument", s);
    }
    MSCS_CHECK_ARG(it.C >= 1 && it.C <= kMaxC && it.rows >= 0, "item %d: C=%d unsupported (1..%d)", s, it.C, kMaxC);
    if (gather) MSCS_CHECK_ARG(it.feat && (kind == kRowsGatherRaw || it.anc_bf16), "item %d: null pointer argument", s);
    else MSCS_CHECK_ARG(it.dF && it.dfeat && it.ldF >= it.C, "item %d: bad gradient arguments", s);
    if (int rc = check_dtype(s, it.dtype, gather ? it.feat : it.dfeat, 1, gather ? "feat" : "dfeat")) return rc;
  }
  return 0;
}

// raw: the items without a normalisation (raw gather; scatter items with anc_f32 == NULL)
template <typename T>
static int rows_launch(const mscs_rows_item* items, int count, RowsKind kind, bool raw, int dtype, cudaStream_t st) {
  RowsBatch g{};
  int blocks = 0;
  for (int s = 0; s < count; ++s) {
    const mscs_rows_item& it = items[s];
    if (it.dtype != dtype || (kind == kRowsScatter && (it.anc_f32 == nullptr) != raw)) continue;
    const int j = g.count++;
    g.feat[j] = it.feat; g.pix[j] = it.pix; g.n_rows_dev[j] = it.n_rows_dev;
    g.bf16[j] = (__nv_bfloat16*)it.anc_bf16; g.f32[j] = it.anc_f32; g.inv[j] = it.inv_norm;
    g.dF[j] = it.dF; g.dfeat[j] = it.dfeat; g.C[j] = it.C; g.ldF[j] = it.ldF; g.rows[j] = it.rows;
    g.block0[j] = blocks;
    blocks += ceil_div(kind == kRowsGather ? (it.rows + 255) / 256 * 256 : it.rows, 8);
  }
  g.block0[g.count] = blocks;
  if (blocks == 0) return 0;
  if (kind == kRowsGather) k_gather_rows_nhwc<T><<<blocks, 256, 0, st>>>(g);
  else if (kind == kRowsGatherRaw) k_rows_raw_nhwc<T, true><<<blocks, 256, 0, st>>>(g);
  else if (raw) k_rows_raw_nhwc<T, false><<<blocks, 256, 0, st>>>(g);
  else k_scatter_rows_nhwc<T><<<blocks, 256, 0, st>>>(g);
  MSCS_LAUNCH_CHECK();
  return 0;
}

static int rows_batch(const mscs_rows_item* items, int count, RowsKind kind, bool raw, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  if (int rc = rows_launch<float>(items, count, kind, raw, MSCS_DTYPE_F32, st)) return rc;
  if (int rc = rows_launch<__nv_bfloat16>(items, count, kind, raw, MSCS_DTYPE_BF16, st)) return rc;
  return rows_launch<__half>(items, count, kind, raw, MSCS_DTYPE_F16, st);
}

extern "C" int mscs_gather_rows_nhwc_batch(const mscs_rows_item* items, int count, void* stream_) {
  if (int rc = rows_check(items, count, kRowsGather)) return rc;
  return rows_batch(items, count, kRowsGather, false, stream_);
}

extern "C" int mscs_gather_raw_rows_batch(const mscs_rows_item* items, int count, void* stream_) {
  if (int rc = rows_check(items, count, kRowsGatherRaw)) return rc;
  return rows_batch(items, count, kRowsGatherRaw, true, stream_);
}

extern "C" int mscs_scatter_rows_nhwc_batch(const mscs_rows_item* items, int count, void* stream_) {
  if (int rc = rows_check(items, count, kRowsScatter)) return rc;
  if (int rc = rows_batch(items, count, kRowsScatter, false, stream_)) return rc;
  return rows_batch(items, count, kRowsScatter, true, stream_);
}
