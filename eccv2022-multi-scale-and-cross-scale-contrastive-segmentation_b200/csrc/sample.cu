// sample.cu -- K1: label down-sampling, per-(image,class) histograms, class-balanced anchor
// selection.  Integer work, bit-exact with the reference:
//   losses/DenseContrastiveLossV2.py:194-206  nearest down-sampling (float32 round trip)
//   losses/DenseContrastiveLossV2.py:86-125   histogram, pair list, per-pair randperm
//   losses/DenseContrastiveLossV2.py:64-84    views-per-class rule
// torch.randperm on the CPU default generator (V2.py:121) = MT19937 + forward Fisher-Yates
// (ATen, third party; restated in oracle/mt19937.py and pinned there against torch itself).
#include "common.cuh"
#include <string.h>

namespace mscs {

constexpr int kTile = 1024;      // pixels per histogram tile
constexpr int kMaxV = 16384;     // views per pair the selection kernel supports

struct ScaleGeo {
  int dl_h, dl_w, hw, tiles;
  int fplane;                    // fh*fw: the flat index y*dl_w+x addresses the flattened FEATURE plane (V2.py:97,123)
  int tile_base;                 // first global tile id of this scale
  int ident_y, ident_x;
  float sy, sx;                  // float(in)/out, as ATen computes it
  size_t off_dlab, off_tilecnt, off_counts, off_kmap, off_pair, off_seg;
  int pair_cap;
};

struct SampleLayout {
  int S, n, H, W, A;
  int ng, b0;                    // pooled mode: images of all ranks / global index of this rank's first image
  ScaleGeo g[MSCS_MAX_SCALES];
  int total_tiles;
  size_t counts_begin, counts_bytes;   // contiguous region holding every scale's counts
  size_t bytes;
};

// pair arrays inside the workspace (per scale, pair_cap entries each)
struct PairArrays {
  int* b; int* c; int* cnt; int* dst; long long* off;
};
__host__ __device__ static inline PairArrays pair_arrays(char* ws, const ScaleGeo& g) {
  PairArrays p;
  char* base = ws + g.off_pair;
  p.off = reinterpret_cast<long long*>(base);
  p.b = reinterpret_cast<int*>(base + sizeof(long long) * g.pair_cap);
  p.c = p.b + g.pair_cap;
  p.cnt = p.c + g.pair_cap;
  p.dst = p.cnt + g.pair_cap;
  return p;
}

static int make_layout(const mscs_sample_cfg* cfg, SampleLayout* L) {
  MSCS_CHECK_ARG(cfg != nullptr, "cfg is null");
  MSCS_CHECK_ARG(cfg->num_scales >= 1 && cfg->num_scales <= MSCS_MAX_SCALES, "num_scales %d out of range",
                 cfg->num_scales);
  MSCS_CHECK_ARG(cfg->n >= 1 && cfg->H >= 1 && cfg->W >= 1, "bad label shape");
  MSCS_CHECK_ARG(cfg->num_classes >= 2 && cfg->num_classes <= 32767, "num_classes %d out of range",
                 cfg->num_classes);
  L->S = cfg->num_scales; L->n = cfg->n; L->H = cfg->H; L->W = cfg->W; L->A = cfg->num_classes;
  L->ng = cfg->n_global > 0 ? cfg->n_global : cfg->n;
  L->b0 = cfg->n_global > 0 ? cfg->image_base : 0;
  MSCS_CHECK_ARG(L->b0 >= 0 && L->b0 + L->n <= L->ng, "image_base/n_global inconsistent");
  size_t off = 0;
  int tile_base = 0;
  // counts first, contiguous, so one memset clears them all
  L->counts_begin = 0;
  for (int s = 0; s < L->S; ++s) {
    L->g[s].off_counts = off;
    off += align_up(sizeof(int) * (size_t)L->n * L->A, 256);
  }
  L->counts_bytes = off;
  for (int s = 0; s < L->S; ++s) {
    ScaleGeo& g = L->g[s];
    MSCS_CHECK_ARG(cfg->fw[s] >= 1 && cfg->fh[s] >= 1, "bad feature size at scale %d", s);
    int scale = cfg->W / cfg->fw[s];                       // V2.py:46 (width only)
    MSCS_CHECK_ARG(scale >= 1, "feature map wider than the label map at scale %d", s);
    g.dl_h = cfg->H / scale; g.dl_w = cfg->W / scale;      // V2.py:205
    MSCS_CHECK_ARG(g.dl_h >= 1 && g.dl_w >= 1, "empty down-sampled label at scale %d", s);
    g.hw = g.dl_h * g.dl_w;
    g.fplane = cfg->fh[s] * cfg->fw[s];
    // the flat index y*dl_w+x addresses the flattened feature plane (V2.py:97,123): it must fit
    MSCS_CHECK_ARG((long long)g.hw <= (long long)cfg->fh[s] * cfg->fw[s],
                   "scale %d: down-sampled label %dx%d exceeds the feature plane %dx%d (the reference would "
                   "index out of range)", s, g.dl_h, g.dl_w, cfg->fh[s], cfg->fw[s]);
    g.tiles = ceil_div(g.hw, kTile);
    g.tile_base = tile_base;
    tile_base += g.tiles * L->n;
    g.ident_y = (g.dl_h == cfg->H); g.ident_x = (g.dl_w == cfg->W);
    g.sy = (float)cfg->H / (float)g.dl_h;
    g.sx = (float)cfg->W / (float)g.dl_w;
    g.pair_cap = L->ng * (L->A - 1);
    g.off_dlab = off;    off += align_up(sizeof(short) * (size_t)L->n * g.hw, 256);
    g.off_tilecnt = off; off += align_up(sizeof(int) * (size_t)L->n * g.tiles * L->A, 256);
    g.off_kmap = off;    off += align_up(sizeof(int) * (size_t)g.pair_cap, 256);
    g.off_pair = off;    off += align_up((sizeof(long long) + 4 * sizeof(int)) * (size_t)g.pair_cap, 256);
    g.off_seg = off;     off += align_up(sizeof(int) * (size_t)(L->A + 1), 256);
  }
  L->total_tiles = tile_base;
  L->bytes = off;
  return 0;
}

// ---------------------------------------------------------------------------------------
// k_label_hist: one CTA per (scale, image, 1024-pixel tile).  Reads the int64 label at the
// nearest-neighbour source position, writes the int16 down-sampled label, a per-tile class
// histogram (for rank->pixel selection) and accumulates the per-image histogram.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ int nearest_src(int dst, float scale, int in_size, int ident) {
  if (ident) return dst;
  int src = (int)floorf(__fmul_rn((float)dst, scale));
  return min(src, in_size - 1);
}

// LabT = long long: the reference's int64 label map; LabT = short: the compact labels of the fused label pass
// (ce.cu:k_label_pass, -1 = outside [0, A)) -- same results, a quarter of the bytes
template <typename LabT>
__global__ void __launch_bounds__(256)
k_label_hist(const __grid_constant__ SampleLayout L, const LabT* __restrict__ labels, char* ws) {
  extern __shared__ int hist[];
  pdl_trigger();
  int t = blockIdx.x;
  int s = 0;
#pragma unroll 1
  for (int i = 1; i < L.S; ++i) if (t >= L.g[i].tile_base) s = i;
  const ScaleGeo& g = L.g[s];
  int local = t - g.tile_base;
  int b = local / g.tiles, tile = local % g.tiles;
  for (int c = threadIdx.x; c < L.A; c += blockDim.x) hist[c] = 0;
  __syncthreads();
  short* dlab = reinterpret_cast<short*>(ws + g.off_dlab) + (size_t)b * g.hw;
  const LabT* lab = labels + (size_t)b * L.H * L.W;
#pragma unroll
  for (int i = 0; i < kTile / 256; ++i) {
    int p = tile * kTile + i * 256 + threadIdx.x;
    if (p < g.hw) {
      int y = p / g.dl_w, x = p - y * g.dl_w;
      int sy = nearest_src(y, g.sy, L.H, g.ident_y);
      int sx = nearest_src(x, g.sx, L.W, g.ident_x);
      long long v = (long long)lab[(size_t)sy * L.W + sx];
      // the reference converts label -> float32 -> int64 (V2.py:205-206)
      float f = (float)v;
      long long c = (long long)f;
      bool ok = (c >= 0 && c < L.A);
      if (ok) atomicAdd(&hist[(int)c], 1);
      dlab[p] = ok ? (short)c : (short)-1;
    }
  }
  __syncthreads();
  int* tilecnt = reinterpret_cast<int*>(ws + g.off_tilecnt) + ((size_t)b * g.tiles + tile) * L.A;
  int* counts = reinterpret_cast<int*>(ws + g.off_counts) + (size_t)b * L.A;
  for (int c = threadIdx.x; c < L.A; c += blockDim.x) {
    int h = hist[c];
    tilecnt[c] = h;
    if (h) atomicAdd(&counts[c], h);
  }
}

// exclusive prefix over the tiles of each (scale, image, class): tilecnt becomes "number of
// class-c pixels of image b before this tile"
__global__ void k_tile_scan(const __grid_constant__ SampleLayout L, char* ws) {
  pdl_trigger();
  pdl_wait();
  int s = blockIdx.y;
  const ScaleGeo& g = L.g[s];
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= L.n * L.A) return;
  int b = e / L.A, c = e - b * L.A;
  int* tc = reinterpret_cast<int*>(ws + g.off_tilecnt) + (size_t)b * g.tiles * L.A + c;
  int run = 0;
  for (int t0 = 0; t0 < g.tiles; t0 += 32) {      // 32 independent loads in flight, then the serial sum
    int v[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = (t0 + i < g.tiles) ? tc[(size_t)(t0 + i) * L.A] : 0;
#pragma unroll
    for (int i = 0; i < 32; ++i)
      if (t0 + i < g.tiles) { tc[(size_t)(t0 + i) * L.A] = run; run += v[i]; }
  }
}

// ---------------------------------------------------------------------------------------
// k_plan: one CTA per scale.  Pair list in torch.where row-major order (V2.py:106), minimum
// count (V2.py:110), views-per-class rule (V2.py:64-84), MT19937 stream offsets (one
// randperm(count) = count-1 draws per pair, V2.py:121), and the class-sorted row layout.
// ---------------------------------------------------------------------------------------
struct PlanCfg { int min_views, max_views, max_total; const int* counts[MSCS_MAX_SCALES]; };

__global__ void __launch_bounds__(1024)
k_plan(const __grid_constant__ SampleLayout L, PlanCfg pc, char* ws, mscs_scale_plan* plan) {
  pdl_wait();
  const int s = blockIdx.x;
  const ScaleGeo& g = L.g[s];
  const int A = L.A, n = L.ng;
  const int* counts = pc.counts[s] ? pc.counts[s] : reinterpret_cast<const int*>(ws + g.off_counts);
  int* kmap = reinterpret_cast<int*>(ws + g.off_kmap);
  int* seg = reinterpret_cast<int*>(ws + g.off_seg);
  PairArrays pa = pair_arrays(ws, g);
  extern __shared__ int npc[];                       // pairs per class, A+1 entries
  __shared__ int warp_pairs[32];
  __shared__ long long warp_draws[32];
  __shared__ int carry_pairs, min_count, single_px;
  __shared__ long long carry_draws;
  __shared__ int sh_V;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  for (int c = tid; c <= A; c += blockDim.x) npc[c] = 0;
  if (tid == 0) { carry_pairs = 0; carry_draws = 0; min_count = 0x7fffffff; single_px = 0; }
  __syncthreads();
  const int entries = n * (A - 1);
  for (int base = 0; base < entries; base += blockDim.x) {
    int e = base + tid;
    int cnt = 0, flag = 0, b = 0, c = 0;
    if (e < entries) {
      b = e / (A - 1); c = e - b * (A - 1);
      cnt = counts[b * A + c];
      flag = cnt >= pc.min_views && cnt > 0;
    }
    // block exclusive scan of (flag, flag ? cnt-1 : 0)
    int pf = flag;
    long long df = flag ? (long long)(cnt - 1) : 0;
    int ps = pf; long long ds = df;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int p2 = __shfl_up_sync(0xffffffffu, ps, o);
      long long d2 = __shfl_up_sync(0xffffffffu, ds, o);
      if (lane >= o) { ps += p2; ds += d2; }
    }
    if (lane == 31) { warp_pairs[wid] = ps; warp_draws[wid] = ds; }
    __syncthreads();
    if (wid == 0) {
      int wp = warp_pairs[lane]; long long wd = warp_draws[lane];
      int wps = wp; long long wds = wd;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int p2 = __shfl_up_sync(0xffffffffu, wps, o);
        long long d2 = __shfl_up_sync(0xffffffffu, wds, o);
        if (lane >= o) { wps += p2; wds += d2; }
      }
      warp_pairs[lane] = wps - wp; warp_draws[lane] = wds - wd;   // exclusive
    }
    __syncthreads();
    int k = carry_pairs + warp_pairs[wid] + ps - pf;
    long long off = carry_draws + warp_draws[wid] + ds - df;
    if (e < entries) kmap[e] = flag ? k : -1;
    if (flag) {
      pa.b[k] = b; pa.c[k] = c; pa.cnt[k] = cnt; pa.off[k] = off;
      atomicMin(&min_count, cnt);
      atomicAdd(&npc[c], 1);
      if (cnt == 1) single_px = 1;
    }
    __syncthreads();
    if (tid == blockDim.x - 1) { carry_pairs = k + pf; carry_draws = off + df; }
    __syncthreads();
  }
  const int T = carry_pairs;
  if (tid == 0) {
    int V = 0, logf = 0;
    if (T > 0) {
      if (pc.max_views == 1) {
        V = min_count;
      } else {
        V = min(min_count, pc.max_views);
        logf = (V == pc.max_views);
      }
      if ((long long)V * T > (long long)pc.max_total) { V = pc.max_total / T; logf = 1; }
    }
    sh_V = V;
    // exclusive scan of pairs-per-class -> class base (in pairs); npc[c] becomes the base
    int run = 0;
    for (int c = 0; c <= A; ++c) { int v = npc[c]; npc[c] = run; run += v; }
    mscs_scale_plan h;
    h.error = (T == 0) ? 1 : (single_px ? 2 : (V > kMaxV ? 3 : 0));
    // on an error the device-driven consumers (selection, gather, similarity forward: they read N from this record
    // before the host has seen it) must find NOTHING to do -- the index arrays are not written then
    h.T = T; h.V = V; h.N = h.error ? 0 : T * V; h.min_count = T > 0 ? min_count : 0; h.log_flag = logf;
    h.dl_h = g.dl_h; h.dl_w = g.dl_w;
    h.draw_base = 0; h.draws = carry_draws;
    plan[s] = h;
  }
  __syncthreads();
  const int V = sh_V;
  for (int c = tid; c <= A; c += blockDim.x) seg[c] = npc[c] * V;
  // rank of each pair inside its class (pairs of one class appear in ascending image order)
  for (int c = tid; c < A - 1; c += blockDim.x) {
    int r = npc[c];
    for (int b = 0; b < n; ++b) {
      int k = kmap[b * (A - 1) + c];
      if (k >= 0) { pa.dst[k] = r * V; ++r; }
    }
  }
}

// ---------------------------------------------------------------------------------------
// k_mt_stream: the raw tempered MT19937 output stream, `total` words, starting at (state,pos).
// One CTA: a 624-word block regenerates in three dependent phases of 227/227/170 words.
// ---------------------------------------------------------------------------------------
struct MtState { uint32_t w[624]; };

__device__ __forceinline__ uint32_t mt_twist(uint32_t u, uint32_t v) {
  uint32_t y = (u & 0x80000000u) | (v & 0x7fffffffu);
  return (y >> 1) ^ ((v & 1u) ? 0x9908b0dfu : 0u);
}
__device__ __forceinline__ uint32_t mt_temper(uint32_t y) {
  y ^= y >> 11; y ^= (y << 7) & 0x9d2c5680u; y ^= (y << 15) & 0xefc60000u; y ^= y >> 18;
  return y;
}

// One CTA on a side stream for 0.2 ms (cfg-2) to 1 ms (pooled cfg-5: 2.8 M words).  It cannot share an SM with a CTA of
// the persistent tensor kernels in any useful way: as a 1024-thread CTA it does not fit next to one (registers), and a
// 128-thread form that does fit is starved of issue slots by the twenty busy warps next to it (0.75 ms at cfg-2) and
// still loses the SM whenever it became resident under the small shared-memory carve-out of the sampling kernels.
// Instead the persistent kernels leave ONE SM free (sim_tc.cuh: persistent_ctas()), which this kernel takes whenever
// it starts; before that, a sweep of 148 CTAs found 147 SMs and took until a second CTA had run on one of them
// (forward stage 0.30 instead of 0.22 ms at cfg-2; sweep 0 of pooled cfg-5 on 8 GPUs 1.31 instead of 0.79 ms).
__global__ void __launch_bounds__(1024)
k_mt_stream(const uint32_t* __restrict__ state, int pos, long long total, uint32_t* __restrict__ out) {
  __shared__ uint32_t buf[2][624];
  const int tid = threadIdx.x;
  for (int i = tid; i < 624; i += 1024) buf[0][i] = state[i];
  __syncthreads();
  // Two warp groups, one barrier per 624-word block:
  //  * threads 0..226 regenerate the NEXT block.  Thread t owns the words t, t+227 and t+454:
  //    new[t] needs only the old block, new[t+227] = new[t] ^ twist(old[t+227], old[t+228]) and
  //    new[t+454] = new[t+227] ^ twist(old[t+454], old[t+455]) chain inside the thread, so the three
  //    dependent phases of the textbook regeneration need no inter-thread synchronisation (word 623
  //    needs new[0], which its owner recomputes);
  //  * threads 256..879 store the CURRENT block meanwhile (one raw word each; tempering is left to
  //    the consumer, which touches only V of the count-1 words of a pair).
  long long produced = 0;
  int first = pos, cur = 0;          // words [first, 624) of buf[cur] are the next outputs
  while (produced < total) {
    const uint32_t* c = buf[cur];
    if (tid < 227) {
      uint32_t* nx = buf[cur ^ 1];
      const uint32_t a = c[tid + 397] ^ mt_twist(c[tid], c[tid + 1]);
      const uint32_t b = a ^ mt_twist(c[tid + 227], c[tid + 228]);
      nx[tid] = a;
      nx[tid + 227] = b;
      if (tid < 169) {
        nx[tid + 454] = b ^ mt_twist(c[tid + 454], c[tid + 455]);
      } else if (tid == 169) {
        const uint32_t n0 = c[397] ^ mt_twist(c[0], c[1]);
        nx[623] = b ^ mt_twist(c[623], n0);
      }
    } else if (tid >= 256) {
      const long long left = total - produced;
      const int n = (int)(left < (long long)(624 - first) ? left : (long long)(624 - first));
      const int j = tid - 256;
      if (j < n) out[produced + j] = c[first + j];      // raw state word: k_fy_select tempers what it uses
    }
    __syncthreads();
    produced += 624 - first;
    first = 0;
    cur ^= 1;
  }
}

// ---------------------------------------------------------------------------------------
// k_fy_select: one CTA per kept pair.  (1) first V steps of the forward Fisher-Yates shuffle
// that torch.randperm(count) performs (only they decide perm[:V], V2.py:121-122) resolved in
// parallel; (2) rank -> pixel: the r-th pixel of class c in image b in raster order
// (= nonzero()[r], V2.py:119) via the per-tile prefix table and a ballot scan of one tile.
// ---------------------------------------------------------------------------------------
struct SelectArgs {
  long long draw_base[MSCS_MAX_SCALES];
  int T[MSCS_MAX_SCALES], V[MSCS_MAX_SCALES];
  int* idx_ref[MSCS_MAX_SCALES];
  int* pair_ref[MSCS_MAX_SCALES];
  int* pix[MSCS_MAX_SCALES];
  int* cls[MSCS_MAX_SCALES];
  int* seg[MSCS_MAX_SCALES];
  int* slot[MSCS_MAX_SCALES];     // optional pixel -> sorted row map (pre-filled with -1 by the caller)
  const mscs_scale_plan* plan_dev; // non-null: T, V and the draw offsets are read from the device plan records
                                   // (the launch then does not wait for the host to have fetched the plan)
};

__global__ void __launch_bounds__(256)
k_fy_select(const __grid_constant__ SampleLayout L, const __grid_constant__ SelectArgs a, char* ws,
            const uint32_t* __restrict__ draws) {
  pdl_trigger();
  pdl_wait();
  const int s = blockIdx.y, k = blockIdx.x;
  int T_s = a.T[s], V_s = a.V[s];
  long long base_s = a.draw_base[s];
  if (a.plan_dev != nullptr) {
    if (a.plan_dev[s].error != 0) return;
    T_s = a.plan_dev[s].T; V_s = a.plan_dev[s].V;
    base_s = 0;
    for (int q = 0; q < s; ++q) base_s += a.plan_dev[q].draws;
  }
  if (k >= T_s) return;
  const ScaleGeo& g = L.g[s];
  const int V = V_s, A = L.A;
  PairArrays pa = pair_arrays(ws, g);
  if (k == 0)                                   // class segments: identical on every rank
    for (int i = threadIdx.x; i <= A; i += blockDim.x) a.seg[s][i] = reinterpret_cast<const int*>(ws + g.off_seg)[i];
  const int bg = pa.b[k], c = pa.c[k], cnt = pa.cnt[k], dst = pa.dst[k];
  const int b = bg - L.b0;                      // local image index
  if (b < 0 || b >= L.n) {
    // another rank's pair (pooled mode): its pixels are not selected here, but the plan is global, so the class id of
    // its sorted rows is known on every rank -- no exchange of the class arrays; pix = -1 marks the rows "not local"
    for (int i = threadIdx.x; i < V; i += blockDim.x) { a.cls[s][dst + i] = c; a.pix[s][dst + i] = -1; }
    if (threadIdx.x == 0) { a.pair_ref[s][2 * k] = bg; a.pair_ref[s][2 * k + 1] = c; }
    return;
  }
  const uint32_t* u = draws + base_s + pa.off[k];
  extern __shared__ int sm[];
  int* t_arr = sm;            // t_i = i + z_i : position swapped with i at step i
  int* w_arr = sm + V;        // w_arr[p] = latest step j < p that wrote position p (t_j == p), or -1
  int* r_arr = sm + 2 * V;    // resolved rank perm[i]
  const int tid = threadIdx.x;
  if (tid == 0) {
    a.pair_ref[s][2 * k] = bg; a.pair_ref[s][2 * k + 1] = c;

  }
  for (int i = tid; i < V; i += blockDim.x) {
    int t = i;
    if (i < cnt - 1) t = i + (int)(mt_temper(u[i]) % (uint32_t)(cnt - i));
    t_arr[i] = t;
    w_arr[i] = -1;
  }
  __syncthreads();
  for (int j = tid; j < V; j += blockDim.x) {
    int t = t_arr[j];
    if (t != j && t < V) atomicMax(&w_arr[t], j);
  }
  __syncthreads();
  for (int i = tid; i < V; i += blockDim.x) {
    const int t = t_arr[i];
    int j1 = -1;
    for (int j = i - 1; j >= 0; --j) if (t_arr[j] == t) { j1 = j; break; }
    int r = t;
    if (j1 >= 0) {                 // position t was last written at step j1 with the value then at j1
      r = j1;
      while (w_arr[r] >= 0) r = w_arr[r];
    }
    r_arr[i] = r;
  }
  __syncthreads();
  // rank -> pixel, one warp per sample.  The per-tile prefix column of (image, class) is staged in
  // smem (t_arr / w_arr are dead by now); the 1024 labels of the hit tile are fetched with 32
  // independent loads per lane-group before the ballots, so one memory latency is paid, not 32.
  const int lane = tid & 31, wid = tid >> 5, nw = blockDim.x >> 5;
  const int* prefix = reinterpret_cast<const int*>(ws + g.off_tilecnt) + (size_t)b * g.tiles * A + c;
  const short* dlab = reinterpret_cast<const short*>(ws + g.off_dlab) + (size_t)b * g.hw;
  int* pre_s = sm;                                  // reuse: needs g.tiles <= 2V ints, else read global
  const bool pre_in_smem = g.tiles <= 2 * V;
  if (pre_in_smem) for (int t = tid; t < g.tiles; t += blockDim.x) pre_s[t] = prefix[(size_t)t * A];
  __syncthreads();
  for (int i = wid; i < V; i += nw) {
    const int r = r_arr[i];
    int lo = 0, hi = g.tiles - 1;          // last tile whose exclusive prefix <= r
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      const int pv = pre_in_smem ? pre_s[mid] : prefix[(size_t)mid * A];
      if (pv <= r) lo = mid; else hi = mid - 1;
    }
    int rem = r - (pre_in_smem ? pre_s[lo] : prefix[(size_t)lo * A]);
    short lab[kTile / 32];
#pragma unroll
    for (int ch = 0; ch < kTile / 32; ++ch) {
      const int q = lo * kTile + ch * 32 + lane;
      lab[ch] = (q < g.hw) ? dlab[q] : (short)-1;
    }
    int p = -1;
#pragma unroll
    for (int ch = 0; ch < kTile / 32; ++ch) {
      const unsigned m = __ballot_sync(0xffffffffu, (int)lab[ch] == c);
      const int pc = __popc(m);
      if (p < 0) {
        if (rem < pc) p = lo * kTile + ch * 32 + (int)__fns(m, 0, rem + 1);
        else rem -= pc;
      }
    }
    if (lane == 0) {
      a.idx_ref[s][(size_t)k * V + i] = p;
      a.pix[s][dst + i] = b * g.fplane + p;      // image base in FEATURE planes: what gather / scatter decode
      a.cls[s][dst + i] = c;
      if (a.slot[s]) a.slot[s][b * g.fplane + p] = dst + i;
    }
  }
}

}  // namespace mscs

using namespace mscs;

extern "C" size_t mscs_sample_workspace_bytes(const mscs_sample_cfg* cfg) {
  SampleLayout L;
  if (make_layout(cfg, &L) != 0) return 0;
  return L.bytes;
}

extern "C" size_t mscs_sample_max_draws(const mscs_sample_cfg* cfg) {
  SampleLayout L;
  if (make_layout(cfg, &L) != 0) return 0;
  size_t d = 0;
  for (int s = 0; s < L.S; ++s) d += (size_t)L.ng * L.g[s].hw;      // the stream covers the pairs of ALL ranks
  return d;
}

extern "C" size_t mscs_sample_counts_offset(const mscs_sample_cfg* cfg, int scale) {
  SampleLayout L;
  if (make_layout(cfg, &L) != 0 || scale < 0 || scale >= L.S) return (size_t)-1;
  return L.g[scale].off_counts;
}

static int sample_hist_any(const mscs_sample_cfg* cfg, const void* labels, bool compact, void* workspace, void* stream_) {
  SampleLayout L;
  int rc = make_layout(cfg, &L);
  if (rc) return rc;
  MSCS_CHECK_ARG(labels && workspace, "null pointer argument");
  cudaStream_t st = (cudaStream_t)stream_;
  char* ws = (char*)workspace;
  MSCS_CUDA(cudaMemsetAsync(ws + L.counts_begin, 0, L.counts_bytes, st));
  if (compact) k_label_hist<short><<<L.total_tiles, 256, sizeof(int) * L.A, st>>>(L, (const short*)labels, ws);
  else k_label_hist<long long><<<L.total_tiles, 256, sizeof(int) * L.A, st>>>(L, (const long long*)labels, ws);
  MSCS_LAUNCH_CHECK();
  dim3 gs(ceil_div(L.n * L.A, 128), L.S);
  MSCS_CUDA(launch_k(k_tile_scan, gs, 128, 0, st, L, ws));
  MSCS_LAUNCH_CHECK();
  return 0;
}

extern "C" int mscs_sample_hist(const mscs_sample_cfg* cfg, const int64_t* labels, void* workspace, void* stream_) {
  return sample_hist_any(cfg, labels, false, workspace, stream_);
}
extern "C" int mscs_sample_hist_i16(const mscs_sample_cfg* cfg, const int16_t* lab16, void* workspace, void* stream_) {
  return sample_hist_any(cfg, lab16, true, workspace, stream_);
}

extern "C" int mscs_sample_plan_from_counts(const mscs_sample_cfg* cfg, const int32_t* const* counts_global,
                                            void* workspace, mscs_scale_plan* plan_dev, void* stream_) {
  SampleLayout L;
  int rc = make_layout(cfg, &L);
  if (rc) return rc;
  MSCS_CHECK_ARG(workspace && plan_dev, "null pointer argument");
  MSCS_CHECK_ARG(cfg->min_views >= 0 && cfg->max_views >= 1 && cfg->max_total >= 1, "bad sampling limits");
  MSCS_CHECK_ARG(L.ng == L.n || counts_global, "pooled mode needs the all-gathered counts");
  PlanCfg pc{cfg->min_views, cfg->max_views, cfg->max_total, {}};
  for (int s = 0; s < L.S; ++s) pc.counts[s] = counts_global ? counts_global[s] : nullptr;
  MSCS_CUDA(launch_k(k_plan, L.S, 1024, sizeof(int) * (L.A + 1), (cudaStream_t)stream_, L, pc, (char*)workspace, plan_dev));
  MSCS_LAUNCH_CHECK();
  return 0;
}

extern "C" int mscs_sample_plan(const mscs_sample_cfg* cfg, const int64_t* labels, void* workspace,
                                mscs_scale_plan* plan_dev, void* stream_) {
  int rc = mscs_sample_hist(cfg, labels, workspace, stream_);
  if (rc) return rc;
  return mscs_sample_plan_from_counts(cfg, nullptr, workspace, plan_dev, stream_);
}
extern "C" int mscs_sample_plan_i16(const mscs_sample_cfg* cfg, const int16_t* lab16, void* workspace,
                                    mscs_scale_plan* plan_dev, void* stream_) {
  int rc = mscs_sample_hist_i16(cfg, lab16, workspace, stream_);
  if (rc) return rc;
  return mscs_sample_plan_from_counts(cfg, nullptr, workspace, plan_dev, stream_);
}

extern "C" int mscs_plan_fetch(const mscs_scale_plan* plan_dev, mscs_scale_plan* plan_host, int num_scales,
                               void* stream_) {
  MSCS_CHECK_ARG(plan_dev && plan_host && num_scales >= 1 && num_scales <= MSCS_MAX_SCALES, "bad arguments");
  cudaStream_t st = (cudaStream_t)stream_;
  MSCS_CUDA(cudaMemcpyAsync(plan_host, plan_dev, sizeof(mscs_scale_plan) * num_scales, cudaMemcpyDeviceToHost, st));
  MSCS_CUDA(cudaStreamSynchronize(st));
  long long base = 0;
  for (int s = 0; s < num_scales; ++s) { plan_host[s].draw_base = base; base += plan_host[s].draws; }
  return 0;
}

extern "C" int mscs_mt19937_stream(const uint32_t* mt_state_host, int mt_pos, uint64_t n_words,
                                   uint32_t* draws_dev, void* stream_) {
  MSCS_CHECK_ARG(mt_state_host && draws_dev, "null pointer argument");
  MSCS_CHECK_ARG(mt_pos >= 0 && mt_pos <= 624, "mt_pos %d out of range", mt_pos);
  cudaStream_t st = (cudaStream_t)stream_;
  if (n_words == 0) return 0;
  // the 624 state words are staged behind the stream (the buffer holds n_words + 1024 words)
  uint32_t* state_dev = draws_dev + align_up((size_t)n_words, 64);
  MSCS_CUDA(cudaMemcpyAsync(state_dev, mt_state_host, sizeof(uint32_t) * 624, cudaMemcpyHostToDevice, st));
  k_mt_stream<<<1, 1024, 0, st>>>(state_dev, mt_pos, (long long)n_words, draws_dev);
  MSCS_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------
// Opt-in counter-based permutation stream (SURVEY.md §8f item 4): Philox4x32-10 (Salmon et al., SC'11), word j of a
// call = philox(counter = (j >> 2, 0, call lo, call hi), key = (seed lo, seed hi))[j & 3].  Random access: no
// sequential generator state, no dependence on the torch CPU generator.  The stream-buffer convention of this
// library is UNTEMPERED MT19937 words (k_fy_select applies the tempering), so the words are stored through the inverse
// tempering: the consumer then sees exactly the Philox outputs (oracle/philox.py) and stays untouched.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t mt_untemper(uint32_t y) {
  y ^= y >> 18;
  y ^= (y << 15) & 0xefc60000u;
  uint32_t t = y;
#pragma unroll
  for (int i = 0; i < 5; ++i) t = y ^ ((t << 7) & 0x9d2c5680u);
  y = t;
#pragma unroll
  for (int i = 0; i < 3; ++i) t = y ^ (t >> 11);
  return t;
}

__device__ __forceinline__ uint4 philox_quad(unsigned long long seed, unsigned long long call, unsigned long long q) {
  uint4 c = make_uint4((uint32_t)q, (uint32_t)(q >> 32), (uint32_t)call, (uint32_t)(call >> 32));
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return make_uint4(mt_untemper(c.x), mt_untemper(c.y), mt_untemper(c.z), mt_untemper(c.w));
}

__global__ void __launch_bounds__(256)
k_philox_stream(unsigned long long seed, unsigned long long call, unsigned long long n_quads, uint4* __restrict__ out) {
  const unsigned long long q = (unsigned long long)blockIdx.x * 256ull + threadIdx.x;
  if (q >= n_quads) return;
  out[q] = philox_quad(seed, call, q);
}

// the call index read from device memory (CUDA graphs: a replay runs the captured launch with its arguments frozen)
__global__ void __launch_bounds__(256) k_philox_stream_dev(unsigned long long seed,
                                                           const unsigned long long* __restrict__ call_dev,
                                                           unsigned long long n_quads, uint4* __restrict__ out) {
  const unsigned long long q = (unsigned long long)blockIdx.x * 256ull + threadIdx.x;
  if (q >= n_quads) return;
  out[q] = philox_quad(seed, *call_dev, q);
}

// next call index: a launch of its own behind the generator on the same stream, i.e. after every reader of the old one
__global__ void k_philox_call_next(unsigned long long* call_dev) { *call_dev += 1ull; }

static int philox_args(const uint32_t* draws_dev, uint64_t n_words) {
  MSCS_CHECK_ARG(draws_dev && ((uintptr_t)draws_dev & 15) == 0, "draws_dev must be a 16-byte aligned device pointer");
  MSCS_CHECK_ARG((n_words + 3) / 4 <= 0x7fffffffull * 256ull, "stream too long");
  return 0;
}

extern "C" int mscs_philox_stream(uint64_t seed, uint64_t call, uint64_t n_words, uint32_t* draws_dev, void* stream_) {
  if (int rc = philox_args(draws_dev, n_words)) return rc;
  if (n_words == 0) return 0;
  const unsigned long long quads = (n_words + 3) / 4;       // the buffer holds n_words rounded up to 4 words
  k_philox_stream<<<(unsigned)((quads + 255) / 256), 256, 0, (cudaStream_t)stream_>>>(seed, call, quads, (uint4*)draws_dev);
  MSCS_LAUNCH_CHECK();
  return 0;
}

extern "C" int mscs_philox_stream_dev(uint64_t seed, uint64_t* call_dev, uint64_t n_words, uint32_t* draws_dev,
                                      void* stream_) {
  MSCS_CHECK_ARG(call_dev && ((uintptr_t)call_dev & 7) == 0, "call_dev must be an 8-byte aligned device pointer");
  if (int rc = philox_args(draws_dev, n_words)) return rc;
  cudaStream_t st = (cudaStream_t)stream_;
  const unsigned long long quads = (n_words + 3) / 4;
  if (quads > 0) {
    k_philox_stream_dev<<<(unsigned)((quads + 255) / 256), 256, 0, st>>>(seed, (const unsigned long long*)call_dev,
                                                                         quads, (uint4*)draws_dev);
    MSCS_LAUNCH_CHECK();
  }
  k_philox_call_next<<<1, 1, 0, st>>>((unsigned long long*)call_dev);
  MSCS_LAUNCH_CHECK();
  return 0;
}

extern "C" int mscs_sample_select(const mscs_sample_cfg* cfg, const mscs_scale_plan* plan_host, void* workspace,
                                  const uint32_t* draws_dev, int32_t* const* idx_ref, int32_t* const* pair_ref,
                                  int32_t* const* pix, int32_t* const* cls, int32_t* const* seg,
                                  int32_t* const* slot, void* stream_) {
  SampleLayout L;
  int rc = make_layout(cfg, &L);
  if (rc) return rc;
  MSCS_CHECK_ARG(plan_host && workspace && draws_dev, "null pointer argument");
  cudaStream_t st = (cudaStream_t)stream_;
  SelectArgs a;
  a.plan_dev = nullptr;
  int maxT = 0, maxV = 0;
  for (int s = 0; s < L.S; ++s) {
    MSCS_CHECK_ARG(plan_host[s].error == 0, "scale %d: sampling plan reports error %d", s, plan_host[s].error);
    MSCS_CHECK_ARG(plan_host[s].V <= kMaxV, "scale %d: %d views per class exceeds the supported %d", s,
                   plan_host[s].V, kMaxV);
    a.draw_base[s] = plan_host[s].draw_base; a.T[s] = plan_host[s].T; a.V[s] = plan_host[s].V;
    a.idx_ref[s] = idx_ref[s]; a.pair_ref[s] = pair_ref[s]; a.pix[s] = pix[s]; a.cls[s] = cls[s]; a.seg[s] = seg[s];
    a.slot[s] = slot ? slot[s] : nullptr;
    if (plan_host[s].T > maxT) maxT = plan_host[s].T;
    if (plan_host[s].V > maxV) maxV = plan_host[s].V;
  }
  size_t smem = sizeof(int) * 3 * (size_t)maxV;
  if (smem > 48 * 1024)
    MSCS_CUDA(cudaFuncSetAttribute(k_fy_select, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid(maxT, L.S);
  k_fy_select<<<grid, 256, smem, st>>>(L, a, (char*)workspace, draws_dev);
  MSCS_LAUNCH_CHECK();
  return 0;
}

// Selection driven by the DEVICE plan records: can be enqueued before the host has seen the plan, so the one
// host synchronisation of the forward pass overlaps this kernel and the gather instead of idling the GPU.
// Grid and shared memory are sized by the configuration's upper bounds (pairs: n_global (A-1); views: v_cap).
extern "C" int mscs_sample_select_async(const mscs_sample_cfg* cfg, const mscs_scale_plan* plan_dev, int v_cap,
                                        void* workspace, const uint32_t* draws_dev, int32_t* const* idx_ref,
                                        int32_t* const* pair_ref, int32_t* const* pix, int32_t* const* cls,
                                        int32_t* const* seg, int32_t* const* slot, void* stream_) {
  SampleLayout L;
  int rc = make_layout(cfg, &L);
  if (rc) return rc;
  MSCS_CHECK_ARG(plan_dev && workspace && draws_dev, "null pointer argument");
  MSCS_CHECK_ARG(v_cap >= 1 && v_cap <= kMaxV, "view bound %d outside 1..%d", v_cap, kMaxV);
  cudaStream_t st = (cudaStream_t)stream_;
  SelectArgs a;
  a.plan_dev = plan_dev;
  for (int s = 0; s < L.S; ++s) {
    a.draw_base[s] = 0; a.T[s] = 0; a.V[s] = 0;
    a.idx_ref[s] = idx_ref[s]; a.pair_ref[s] = pair_ref[s]; a.pix[s] = pix[s]; a.cls[s] = cls[s]; a.seg[s] = seg[s];
    a.slot[s] = slot ? slot[s] : nullptr;
  }
  const int n_glob = cfg->n_global > 0 ? cfg->n_global : cfg->n;
  const int t_cap = n_glob * (cfg->num_classes - 1);
  size_t smem = sizeof(int) * 3 * (size_t)v_cap;
  if (smem > 48 * 1024)
    MSCS_CUDA(cudaFuncSetAttribute(k_fy_select, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid(t_cap, L.S);
  MSCS_CUDA(launch_k(k_fy_select, grid, 256, smem, st, L, a, (char*)workspace, draws_dev));
  MSCS_LAUNCH_CHECK();
  return 0;
}

// Split plan fetch: begin = async D2H into a pinned staging buffer + event; end = wait for that event only
// (work enqueued after begin keeps running) and hand the records out.  The copy runs on a private stream that
// waits for the producer stream's position at the call: the producer stream itself (selection kernel next) does
// not queue behind the copy.
// One set of resources per (host thread, device): a process that drives several GPUs from one thread must not
// record on a stream that belongs to another device.
constexpr int kMaxDevices = 64;
struct PlanFetch { mscs_scale_plan* pinned; cudaEvent_t done, src; cudaStream_t stream; };
static thread_local PlanFetch t_fetch[kMaxDevices] = {};
static thread_local int t_fetch_dev = -1;      // device of the outstanding fetch
extern "C" int mscs_plan_fetch_begin(const mscs_scale_plan* plan_dev, int num_scales, void* stream_) {
  MSCS_CHECK_ARG(plan_dev && num_scales >= 1 && num_scales <= MSCS_MAX_SCALES, "bad arguments");
  cudaStream_t st = (cudaStream_t)stream_;
  int dev = 0;
  MSCS_CUDA(cudaGetDevice(&dev));
  MSCS_CHECK_ARG(dev >= 0 && dev < kMaxDevices, "device ordinal %d out of range", dev);
  PlanFetch& f = t_fetch[dev];
  if (!f.pinned) {
    MSCS_CUDA(cudaHostAlloc((void**)&f.pinned, sizeof(mscs_scale_plan) * MSCS_MAX_SCALES, cudaHostAllocDefault));
    MSCS_CUDA(cudaEventCreateWithFlags(&f.done, cudaEventDisableTiming));
    MSCS_CUDA(cudaEventCreateWithFlags(&f.src, cudaEventDisableTiming));
    int lo = 0, hi = 0;
    MSCS_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    MSCS_CUDA(cudaStreamCreateWithPriority(&f.stream, cudaStreamNonBlocking, hi));
  }
  MSCS_CUDA(cudaEventRecord(f.src, st));
  MSCS_CUDA(cudaStreamWaitEvent(f.stream, f.src, 0));
  MSCS_CUDA(cudaMemcpyAsync(f.pinned, plan_dev, sizeof(mscs_scale_plan) * num_scales, cudaMemcpyDeviceToHost,
                            f.stream));
  MSCS_CUDA(cudaEventRecord(f.done, f.stream));
  t_fetch_dev = dev;
  return 0;
}
extern "C" int mscs_plan_fetch_end(mscs_scale_plan* plan_host, int num_scales) {
  MSCS_CHECK_ARG(plan_host && num_scales >= 1 && num_scales <= MSCS_MAX_SCALES, "bad arguments");
  MSCS_CHECK_ARG(t_fetch_dev >= 0, "mscs_plan_fetch_end without mscs_plan_fetch_begin on this thread");
  PlanFetch& f = t_fetch[t_fetch_dev];
  MSCS_CUDA(cudaEventSynchronize(f.done));
  long long base = 0;
  for (int s = 0; s < num_scales; ++s) {
    plan_host[s] = f.pinned[s];
    plan_host[s].draw_base = base; base += plan_host[s].draws;
  }
  return 0;
}

static inline uint32_t host_twist(uint32_t u, uint32_t v) {
  const uint32_t y = (u & 0x80000000u) | (v & 0x7fffffffu);
  return (y >> 1) ^ ((0u - (v & 1u)) & 0x9908b0dfu);
}
// one block regeneration in the three-phase form (old -> new buffer) so the compiler vectorises it
__attribute__((target_clones("avx2", "default")))
static void host_regen(const uint32_t* __restrict__ o, uint32_t* __restrict__ n) {
#pragma GCC ivdep
  for (int i = 0; i < 227; ++i) n[i] = o[i + 397] ^ host_twist(o[i], o[i + 1]);
#pragma GCC ivdep
  for (int i = 0; i < 227; ++i) n[227 + i] = n[i] ^ host_twist(o[227 + i], o[228 + i]);
#pragma GCC ivdep
  for (int i = 0; i < 169; ++i) n[454 + i] = n[227 + i] ^ host_twist(o[454 + i], o[455 + i]);
  n[623] = n[396] ^ host_twist(o[623], n[0]);
}

extern "C" int mscs_mt19937_advance_host(uint32_t* mt, int* pos, uint64_t k) {
  MSCS_CHECK_ARG(mt && pos && *pos >= 0 && *pos <= 624, "bad MT19937 state");
  uint32_t buf[2][624];
  memcpy(buf[0], mt, sizeof(buf[0]));
  int cur = 0, p = *pos;
  while (k > 0) {
    if (p >= 624) { host_regen(buf[cur], buf[cur ^ 1]); cur ^= 1; p = 0; }
    const uint64_t take = (uint64_t)(624 - p) < k ? (uint64_t)(624 - p) : k;
    p += (int)take;
    k -= take;
  }
  memcpy(mt, buf[cur], sizeof(buf[0]));
  *pos = p;
  return 0;
}
