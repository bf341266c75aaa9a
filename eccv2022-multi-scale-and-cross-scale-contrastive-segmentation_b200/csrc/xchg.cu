// xchg.cu -- pooled cross-batch mode: the data-plane exchange between the GPUs of one box, done by OUR kernels over
// NVLink peer memory instead of collectives on zero-initialised slabs.
//
// The reference evaluates the loss per rank on its local images (utils/distributed.py:63-73 `concat_all_gather` is
// imported by DenseContrastiveLossV2_ms.py:3 but never called); the pooled mode north_star adds contrasts the anchors
// of ALL ranks.  Every rank owns one "exchange slab" (cudaMalloc + CUDA IPC: every peer maps it), laid out identically
// on every rank: flags | per step parity: operand matrices (bf16) | row statistics | gradient rows.
//
//   k_gather_p2p        K2 fused with the all-gather: every normalised bf16 anchor row is stored -- 16 bytes per lane,
//                       one 512-byte row per warp instruction -- straight into the SAME sorted row of the operand
//                       matrix of every rank (its own included).  No packing, no collective, no zero slab.
//   k_gather_rows_p2p   the same for channels-last maps: one warp per sorted row of this rank.
//   k_push_ranges       row statistics of this rank's anchor-row range (accumulated in PRIVATE memory: the sweeps'
//                       per-tile atomics into the peer-mapped slab itself ran sweep 0 1.7x slower) -> the same rows
//                       of every rank's slab.
//   k_xchg_barrier      release/acquire flag barrier across the ranks (one flag word per rank, monotonic epoch):
//                       orders "my stores have landed everywhere" before "I read what the others stored".
//   scatter (pull)      gather.cu: the scatter reads every gradient row from the rank that computed it.
// Slabs are double-buffered by step parity, so a rank that runs ahead never writes into a buffer a slower rank is
// still reading (DESIGN.md section 6 has the argument).
#include "rows.cuh"

namespace mscs {

struct PeerPtrs { void* p[MSCS_MAX_RANKS]; int n; };

__device__ __forceinline__ unsigned long long xg_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// flags[r] of every rank's slab: the epoch rank r has reached.  Thread r publishes this rank's epoch on peer r and
// waits until peer r's epoch has arrived here.  Monotonic epochs: a rank that is already one barrier ahead only makes
// the comparison (>=) true earlier.  A wait that lasts longer than `timeout_ns` traps (a missing rank must surface as
// a launch error, not hang the GPU).
__global__ void k_xchg_barrier(PeerPtrs flags, int rank, uint32_t epoch, unsigned long long timeout_ns) {
  const int r = threadIdx.x;
  if (r >= flags.n) return;
  __threadfence_system();
  st_release_sys(reinterpret_cast<uint32_t*>(flags.p[r]) + rank, epoch);
  const uint32_t* mine = reinterpret_cast<const uint32_t*>(flags.p[rank]) + r;
  const unsigned long long t0 = xg_timer_ns();
  while ((int32_t)(ld_acquire_sys(mine) - epoch) < 0) {
    if (xg_timer_ns() - t0 > timeout_ns) __trap();
    __nanosleep(200);
  }
  __threadfence_system();
}

// up to 48 ranges per call: copy len[j] floats from src + src_off[j] (private memory of this rank) to float offset
// off[j] of EVERY rank's slab, this rank's own included
struct PushArgs { PeerPtrs slab; const float* src; int count; long long off[48]; long long src_off[48]; int len[48]; };
__global__ void __launch_bounds__(256) k_push_ranges(const __grid_constant__ PushArgs a) {
  const int j = blockIdx.y;
  if (j >= a.count) return;
  const float* src = a.src + a.src_off[j];
  const int len = a.len[j];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < len; i += gridDim.x * blockDim.x) {
    const float v = src[i];
    for (int r = 0; r < a.slab.n; ++r) reinterpret_cast<float*>(a.slab.p[r])[a.off[j] + i] = v;
  }
}

// K2 + all-gather.  One warp per 8-pixel octet of the slot map (address order, like k_gather_sectors_batch); lane l
// owns channels [8l, 8l+8): eight strided sector reads, then ONE 16-byte store per destination matrix.
struct GatherP2P {
  const void* feat; const int* slot; float* anc_f32; float* inv_norm;
  PeerPtrs bf16;            // the operand matrix of this scale in every rank's slab (same sorted row index everywhere)
  int C, C_pad, plane, n_octets, rank;
  int n_rows;               // N: the local padding rows [N, N_pad) are zeroed by the extra last block
  const int* n_rows_dev;    // optional: N lives in device memory (the launch then does not wait for the host)
};
// T: element type of the map (float / bf16 / fp16).  Loads widen exactly to fp32 (to_f32) and everything after them is
// the fp32 arithmetic, so a half map gives the rows of its fp32 widening bit for bit.
template <typename T>
__global__ void __launch_bounds__(256) k_gather_p2p(const __grid_constant__ GatherP2P g) {
  const int lane = threadIdx.x & 31;
  if (blockIdx.x == gridDim.x - 1) {      // padding rows of the LOCAL matrix (the TMA tiles read them)
    const int N = g.n_rows_dev ? *g.n_rows_dev : g.n_rows, N_pad = (N + 255) / 256 * 256;
    uint32_t* z = reinterpret_cast<uint32_t*>(reinterpret_cast<__nv_bfloat16*>(g.bf16.p[g.rank]) + (size_t)N * g.C_pad);
    for (int i = threadIdx.x; i < (N_pad - N) * (g.C_pad / 2); i += blockDim.x) z[i] = 0u;
    return;
  }
  const int oct = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (oct >= g.n_octets) return;
  const int gp = oct * 8;
  const int s_mine = (lane < 8) ? g.slot[gp + lane] : -1;
  unsigned act = __ballot_sync(0xffffffffu, s_mine >= 0);
  if (act == 0) return;
  const int C = g.C, plane = g.plane;
  const int b = gp / plane, p = gp - b * plane;
  const T* src0 = static_cast<const T*>(g.feat) + ((size_t)b * C) * plane + p;
  const int c0 = lane * 8;
  while (act) {
    const int j = __ffs(act) - 1;
    act &= act - 1;
    const int row = __shfl_sync(0xffffffffu, s_mine, j);
    const T* src = src0 + j;
    float v[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) v[q] = (c0 + q < C) ? to_f32(__ldg(src + (size_t)(c0 + q) * plane)) : 0.f;
    const float inv = inv_norm_of(v);
    if (lane == 0) g.inv_norm[row] = inv;
    uint32_t pk[4];
#pragma unroll
    for (int q = 0; q < 8; q += 2) {
      const float f0 = v[q] * inv, f1 = v[q + 1] * inv;
      if (c0 + q < C) g.anc_f32[(size_t)row * C + c0 + q] = f0;
      if (c0 + q + 1 < C) g.anc_f32[(size_t)row * C + c0 + q + 1] = f1;
      __nv_bfloat162 h = __floats2bfloat162_rn(f0, f1);      // channels >= C hold exact zeros (v = 0)
      pk[q >> 1] = *reinterpret_cast<uint32_t*>(&h);
    }
    if (c0 < g.C_pad) {
      const uint4 w = make_uint4(pk[0], pk[1], pk[2], pk[3]);
      for (int r = 0; r < g.bf16.n; ++r)
        *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(g.bf16.p[r]) + (size_t)row * g.C_pad + c0) = w;
    }
  }
}

// Channels-last maps: one warp per sorted row with pix >= 0; lane l owns the channels l + 32 q, the lane / channel
// assignment of k_gather_rows_nhwc, so the unit rows, inverse norms and operand rows equal the single-process ones bit
// for bit.  The fp32 row and inverse norm stay local, the bf16 row is stored into every rank's operand matrix.
// Rows with pix < 0 are NOT written: they belong to other ranks, whose peer stores land in this slab concurrently.
// Only the local padding rows [N, N_pad) are zeroed.
struct GatherRowsP2P {
  const void* feat; const int* pix; float* anc_f32; float* inv_norm;
  PeerPtrs bf16;            // as GatherP2P
  int C, C_pad, rank;
  int n_rows;               // N, or its upper bound when n_rows_dev is set (sizes the grid)
  const int* n_rows_dev;
};
template <typename T>
__global__ void __launch_bounds__(256) k_gather_rows_p2p(const __grid_constant__ GatherRowsP2P g) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int N = g.n_rows_dev ? *g.n_rows_dev : g.n_rows, N_pad = (N + 255) / 256 * 256;
  if (row >= N_pad) return;
  const int C = g.C, C_pad = g.C_pad;
  if (row >= N) {
    __nv_bfloat16* orow = reinterpret_cast<__nv_bfloat16*>(g.bf16.p[g.rank]) + (size_t)row * C_pad;
    for (int c = lane; c < C_pad; c += 32) orow[c] = __float2bfloat16(0.f);
    return;
  }
  const int gp = g.pix[row];
  if (gp < 0) return;
  const T* src = static_cast<const T*>(g.feat) + (size_t)gp * C;
  float v[kMaxC / 32];
#pragma unroll
  for (int q = 0; q < kMaxC / 32; ++q) {
    const int c = lane + 32 * q;
    v[q] = (c < C) ? to_f32(__ldg(src + c)) : 0.f;
  }
  const float inv = inv_norm_of(v);
  if (lane == 0) g.inv_norm[row] = inv;
  store_unit_row(v, inv, C, C_pad, g.anc_f32 + (size_t)row * C, [&](int c, __nv_bfloat16 h) {
    for (int r = 0; r < g.bf16.n; ++r) reinterpret_cast<__nv_bfloat16*>(g.bf16.p[r])[(size_t)row * C_pad + c] = h;
  });
}

// Projector tail in the pooled mode: this rank's rows in compact order.  One CTA per scale scans the sorted rows 1024
// at a time; a row below the device count with pix >= 0 is local and gets k = the number of local rows before it, so
// the compact order is the global row order restricted to the local rows (no atomics: deterministic).
struct LocalRows {
  const int* pix[MSCS_MAX_SCALES]; const int* n_rows_dev[MSCS_MAX_SCALES]; int* crow[MSCS_MAX_SCALES];
  int* cpix[MSCS_MAX_SCALES]; int* slot[MSCS_MAX_SCALES]; int rows[MSCS_MAX_SCALES]; int* n_local_dev;
};
__global__ void __launch_bounds__(1024) k_local_rows(const __grid_constant__ LocalRows a) {
  const int s = blockIdx.x;
  const int* __restrict__ pix = a.pix[s];
  int* __restrict__ crow = a.crow[s];
  int* __restrict__ cpix = a.cpix[s];
  int* __restrict__ slot = a.slot[s];
  const int rows = a.rows[s];
  __shared__ int warp_total[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int N = max(0, min(*a.n_rows_dev[s], rows));      // pix entries at and above the count are stale
  int base = 0;
  for (int r0 = 0; r0 < rows; r0 += 1024) {
    const int r = r0 + (int)threadIdx.x;
    const int p = r < N ? pix[r] : -1;
    const unsigned m = __ballot_sync(0xffffffffu, p >= 0);
    if (lane == 0) warp_total[warp] = __popc(m);
    __syncthreads();
    int before = 0, total = 0;
    for (int w = 0; w < 32; ++w) {
      const int t = warp_total[w];
      before += w < warp ? t : 0;
      total += t;
    }
    const int k = base + before + __popc(m & ((1u << lane) - 1u));
    if (r < rows) crow[r] = p >= 0 ? k : -1;
    if (p >= 0) {
      cpix[k] = p;
      if (slot) slot[p] = k;
    }
    base += total;
    __syncthreads();      // warp_total is rewritten by the next chunk
  }
  if (threadIdx.x == 0) a.n_local_dev[s] = base;
}

}  // namespace mscs

using namespace mscs;

extern "C" int mscs_local_rows_batch(const int32_t* const* pix, const int32_t* const* n_rows_dev, const int32_t* rows,
                                     int32_t* const* crow, int32_t* const* cpix, int32_t* const* slot,
                                     int32_t* n_local_dev, int count, void* stream_) {
  MSCS_CHECK_ARG(count >= 1 && count <= MSCS_MAX_SCALES, "bad scale count %d", count);
  MSCS_CHECK_ARG(pix && n_rows_dev && rows && crow && cpix && n_local_dev, "null pointer argument");
  MSCS_CHECK_ARG((uintptr_t)n_local_dev % 4 == 0, "n_local_dev must be 4-byte aligned");
  LocalRows a{};
  a.n_local_dev = n_local_dev;
  for (int s = 0; s < count; ++s) {
    MSCS_CHECK_ARG(pix[s] && n_rows_dev[s] && crow[s] && cpix[s], "scale %d: null pointer argument", s);
    MSCS_CHECK_ARG(rows[s] >= 0, "scale %d: %d rows", s, rows[s]);
    const int32_t* sl = slot ? slot[s] : nullptr;
    for (const void* p : {(const void*)pix[s], (const void*)n_rows_dev[s], (const void*)crow[s], (const void*)cpix[s],
                          (const void*)sl})
      MSCS_CHECK_ARG((uintptr_t)p % 4 == 0, "scale %d: int32 arrays must be 4-byte aligned", s);
    a.pix[s] = pix[s]; a.n_rows_dev[s] = n_rows_dev[s]; a.crow[s] = crow[s]; a.cpix[s] = cpix[s];
    a.slot[s] = const_cast<int*>(sl); a.rows[s] = rows[s];
  }
  k_local_rows<<<count, 1024, 0, (cudaStream_t)stream_>>>(a);
  MSCS_LAUNCH_CHECK();
  return 0;
}

static int fill_peers(PeerPtrs* out, void* const* ptrs, int n, size_t byte_off) {
  MSCS_CHECK_ARG(ptrs && n >= 1 && n <= MSCS_MAX_RANKS, "bad peer table (%d ranks, at most %d)", n, MSCS_MAX_RANKS);
  out->n = n;
  for (int r = 0; r < n; ++r) {
    MSCS_CHECK_ARG(ptrs[r] != nullptr, "peer %d: null slab pointer", r);
    out->p[r] = (char*)ptrs[r] + byte_off;
  }
  return 0;
}

extern "C" int mscs_xchg_alloc(size_t bytes, void** dev_ptr, unsigned char* handle_out) {
  MSCS_CHECK_ARG(bytes > 0 && dev_ptr && handle_out, "bad arguments");
  void* p = nullptr;
  MSCS_CUDA(cudaMalloc(&p, bytes));
  MSCS_CUDA(cudaMemset(p, 0, bytes));
  cudaIpcMemHandle_t h;
  MSCS_CUDA(cudaIpcGetMemHandle(&h, p));
  static_assert(sizeof(h) == MSCS_IPC_HANDLE_BYTES, "IPC handle size");
  memcpy(handle_out, &h, sizeof(h));
  MSCS_CUDA(cudaDeviceSynchronize());
  *dev_ptr = p;
  return 0;
}

extern "C" int mscs_xchg_open(const unsigned char* handle, void** dev_ptr) {
  MSCS_CHECK_ARG(handle && dev_ptr, "bad arguments");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  MSCS_CUDA(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return 0;
}

extern "C" int mscs_xchg_close(void* dev_ptr) {
  if (dev_ptr) MSCS_CUDA(cudaIpcCloseMemHandle(dev_ptr));
  return 0;
}

extern "C" int mscs_xchg_free(void* dev_ptr) {
  if (dev_ptr) MSCS_CUDA(cudaFree(dev_ptr));
  return 0;
}

extern "C" int mscs_xchg_barrier(void* const* slabs, int world, int rank, uint32_t epoch, double timeout_s, void* stream_) {
  PeerPtrs f;
  if (int rc = fill_peers(&f, slabs, world, 0)) return rc;
  MSCS_CHECK_ARG(rank >= 0 && rank < world && epoch > 0, "bad rank / epoch");
  const unsigned long long ns = (unsigned long long)((timeout_s > 0 ? timeout_s : 20.0) * 1e9);
  k_xchg_barrier<<<1, 32, 0, (cudaStream_t)stream_>>>(f, rank, epoch, ns);
  MSCS_LAUNCH_CHECK();
  return 0;
}

extern "C" int mscs_xchg_push(void* const* slabs, int world, const float* src, const int64_t* src_float_off,
                              const int64_t* float_off, const int32_t* len, int count, void* stream_) {
  MSCS_CHECK_ARG(src && src_float_off && float_off && len && count >= 0 && count <= 48,
                 "bad range list (%d ranges, at most 48)", count);
  if (count == 0) return 0;
  PushArgs a{};
  if (int rc = fill_peers(&a.slab, slabs, world, 0)) return rc;
  a.src = src; a.count = count;
  int maxlen = 0;
  for (int j = 0; j < count; ++j) {
    a.off[j] = float_off[j]; a.src_off[j] = src_float_off[j]; a.len[j] = len[j];
    if (len[j] > maxlen) maxlen = len[j];
  }
  if (maxlen == 0) return 0;
  const int bx = ceil_div(maxlen, 256) < 64 ? ceil_div(maxlen, 256) : 64;
  k_push_ranges<<<dim3(bx, count), 256, 0, (cudaStream_t)stream_>>>(a);
  MSCS_LAUNCH_CHECK();
  return 0;
}

extern "C" int mscs_gather_normalize_p2p(const void* feat, int n, int C, int plane, const int32_t* slot, int N,
                                         const int32_t* n_rows_dev, void* const* slabs, int world, int rank,
                                         size_t bf16_byte_off, float* anc_f32, float* inv_norm, void* stream_, int dtype) {
  MSCS_CHECK_ARG(feat && slot && anc_f32 && inv_norm, "null pointer argument");
  MSCS_CHECK_ARG(C >= 1 && C <= kMaxC && plane % 8 == 0 && n >= 1 && N >= 0, "unsupported shape (C %d, plane %d)", C, plane);
  MSCS_CHECK_ARG(rank >= 0 && rank < world && bf16_byte_off % 16 == 0, "bad rank / offset");
  if (int rc = check_dtype(-1, dtype, feat, 1, "feat")) return rc;
  GatherP2P g{};
  if (int rc = fill_peers(&g.bf16, slabs, world, bf16_byte_off)) return rc;
  g.feat = feat; g.slot = slot; g.anc_f32 = anc_f32; g.inv_norm = inv_norm;
  g.C = C; g.C_pad = (C + 63) / 64 * 64; g.plane = plane; g.n_octets = n * plane / 8; g.rank = rank; g.n_rows = N; g.n_rows_dev = n_rows_dev;
  const int grid = ceil_div(g.n_octets, 8) + 1;
  cudaStream_t st = (cudaStream_t)stream_;
  if (dtype == MSCS_DTYPE_F32) k_gather_p2p<float><<<grid, 256, 0, st>>>(g);
  else if (dtype == MSCS_DTYPE_BF16) k_gather_p2p<__nv_bfloat16><<<grid, 256, 0, st>>>(g);
  else k_gather_p2p<__half><<<grid, 256, 0, st>>>(g);
  MSCS_LAUNCH_CHECK();
  return 0;
}

extern "C" int mscs_gather_rows_p2p(const void* feat, int C, const int32_t* pix, int N, const int32_t* n_rows_dev,
                                    void* const* slabs, int world, int rank, size_t bf16_byte_off, float* anc_f32,
                                    float* inv_norm, void* stream_, int dtype) {
  MSCS_CHECK_ARG(feat && pix && anc_f32 && inv_norm, "null pointer argument");
  MSCS_CHECK_ARG(C >= 1 && C <= kMaxC && N >= 0, "unsupported shape (C %d, %d rows)", C, N);
  MSCS_CHECK_ARG(rank >= 0 && rank < world && bf16_byte_off % 16 == 0, "bad rank / offset");
  if (int rc = check_dtype(-1, dtype, feat, 1, "feat")) return rc;
  GatherRowsP2P g{};
  if (int rc = fill_peers(&g.bf16, slabs, world, bf16_byte_off)) return rc;
  g.feat = feat; g.pix = pix; g.anc_f32 = anc_f32; g.inv_norm = inv_norm;
  g.C = C; g.C_pad = (C + 63) / 64 * 64; g.rank = rank; g.n_rows = N; g.n_rows_dev = n_rows_dev;
  const int grid = ceil_div((N + 255) / 256 * 256, 8);
  if (grid == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream_;
  if (dtype == MSCS_DTYPE_F32) k_gather_rows_p2p<float><<<grid, 256, 0, st>>>(g);
  else if (dtype == MSCS_DTYPE_BF16) k_gather_rows_p2p<__nv_bfloat16><<<grid, 256, 0, st>>>(g);
  else k_gather_rows_p2p<__half><<<grid, 256, 0, st>>>(g);
  MSCS_LAUNCH_CHECK();
  return 0;
}
