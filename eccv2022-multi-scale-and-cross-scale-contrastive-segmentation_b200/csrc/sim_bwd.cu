// sim_bwd.cu -- K4 (tensor half): fused backward of the similarity / loss, recomputing logit
// tiles instead of storing them.  Replaces the autograd backward of V2.py:138-188 and
// _ms.py:95-156 up to d loss / d (unit rows); the normalisation backward + dense scatter is
// gather.cu.
//
// One pass computes  dX_rows += scale * W(rows, cols) * Y_cols  with
//   W_ij = E_ij (cS_i + cS_j)                                   (negative pair)
//   W_ij = -( cPN_i / (E_ij + neg_i) + cPN_j / (E_ij + neg_j) ) (positive pair, 0 on the diagonal)
// where cS = S/(div N1), cPN = neg/(div N1) come from the forward (k_finalize).  A single-scale
// term is ONE pass with both the row and column coefficients (W = G + G^T, so no second product);
// a cross-scale term is a pass with row coefficients only (dA) and, unless the key side is
// detached, a pass with rows = keys and column coefficients only (dK).
//
// CTA = 128 rows x a run of 128-column units; a unit is processed as two 64-column tiles.
//   X rows (the A operand of every S MMA of the run) live in TENSOR MEMORY for the whole run
//   (written once per run with tcgen05.st), so shared memory holds nothing but a 3-stage ring of
//   Y units (64 KB each): a unit is requested two units (~4000 cycles) before its first MMA.
// Per 64-column tile:
//   MMA 1  S = X Y^T   (A from TMEM, B K-major from smem, N = 64)   -> TMEM, double buffered
//   epilogue: W = f(exp2(S)) as packed bf16 written back INTO the S columns of TMEM (in place)
//   MMA 2  dX += W Y   (A = W from TMEM; the same Y rows as an MN-major B operand, N = C_pad) -> TMEM
// dX stays in TMEM for the whole run and is flushed with fp32 reductions at the end.
// TMEM columns: dX [0,256) | X [256,384) | S/W buffers [384,448), [448,512).
// (History: with X and two Y stages in smem the MMA warp waited for TMA data 43% of the time -- a
// stage was refilled only when the dX product of the same stage had finished, so the ~1 us TMA
// round trip was exposed on every tile; see DESIGN.md.)
#include "sim_tc.cuh"
#include <stdlib.h>

namespace mscs {

constexpr int kBwdEpiWarps = 16;     // 4 per SM sub-partition: thread = (row, 16-column quarter of a tile).  The
                                     // S -> W conversion sits between the two MMAs of a tile (S buffer cycle =
                                     // S MMAs + conversion + dX MMAs), so its LATENCY bounds the tile rate
constexpr int kBwdThreads = 128 + 32 * kBwdEpiWarps;
constexpr int kBwdStages = 3;
constexpr int kBwdSub = 64;          // columns per tile (half a unit)
constexpr uint32_t kTmX = 256, kTmS = 384;

struct BwdDev {
  const int* row_cls; const int* col_seg;
  const float* row_cs; const float* row_cpn; const float* row_neg;
  const float* col_cs; const float* col_cpn; const float* col_neg;
  const __nv_bfloat16* x_rows;      // (N_pad, C_pad) row operand matrix (read directly into TMEM)
  float* dF; int ld;
  int n_rows, n_cols, self_mask, y_map;
  float scale_log2, out_scale;
};
struct BwdArgs {
  alignas(64) CUtensorMap maps[MSCS_MAX_SCALES];
  BwdDev p[MSCS_MAX_PASSES];
  WorkTable work;
  const float* grad_out;
  // DEV instance only: device-resident row / column counts of every pass (n_rows / n_cols are then upper bounds).
  // Kept behind every field the eager instance reads, so that instance compiles as it did without them.
  const int* rows_dev[MSCS_MAX_PASSES]; const int* cols_dev[MSCS_MAX_PASSES];
};

__host__ __device__ constexpr size_t bwd_smem_bytes(int KB) {
  return 1024 + (size_t)(kBwdStages * KB) * kBlkBytes + (size_t)kBwdEpiWarps * 2 * 3 * 32 * sizeof(float) + 256;
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d)
               : "memory");
}

// DEV: the row and column counts of a pass are read from device memory (args.rows_dev / cols_dev, written by the
// sampling plan of the same step) once per run, after the PDL wait; rows and columns beyond them -- stale data of
// earlier calls inside the upper bounds -- are treated exactly like the padding beyond n_rows / n_cols
template <int KB, bool DEV>
__global__ void __launch_bounds__(kBwdThreads, 1) k_sim_bwd(const __grid_constant__ BwdArgs args) {
  constexpr int CP = KB * 64;                       // padded channel count = N of the second MMA
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smB = smem;                                         // [stages][KB][128 rows][128 B] Y units
  float* cstat = reinterpret_cast<float*>(smB + (size_t)kBwdStages * KB * kBlkBytes);   // per epilogue warp: [2][3][32]
  uint64_t* bars = reinterpret_cast<uint64_t*>(cstat + kBwdEpiWarps * 2 * 3 * 32);
  uint64_t* b_full = bars;                    // [stages] (one barrier per unit: the ring is deep enough)
  uint64_t* b_empty = bars + 12;              // [stages]
  uint64_t* s_full = bars + 15;               // [2]
  uint64_t* w_full = bars + 17;               // [2]
  uint64_t* df_full = bars + 19;  uint64_t* df_empty = bars + 20;
  uint64_t* x_full = bars + 21;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 22);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_trigger();
  if (warp == 0 && lane == 0) {
    for (int i = 0; i < kBwdStages; ++i) {
      ptx::mbar_init(&b_full[i], 1);
      ptx::mbar_init(&b_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) { ptx::mbar_init(&s_full[i], 1); ptx::mbar_init(&w_full[i], kBwdEpiWarps); }
    ptx::mbar_init(df_full, 1); ptx::mbar_init(df_empty, kBwdEpiWarps);
    ptx::mbar_init(x_full, kBwdEpiWarps);
    ptx::fence_barrier_init();
  }
  if (warp == 2) ptx::tmem_alloc(tmem_slot, 512);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();       // barriers and tensor memory are set up while the previous grid (work-table build) drains
#if defined(MSCS_WAIT_PROFILE) || defined(MSCS_TRACE)     // effective SM clock of this launch: slot 31 accumulates (ns, cycles) of CTA 0
  const unsigned long long prof_t0 = ptx::globaltimer_ns();
  const long long prof_c0 = clock64();
  (void)prof_t0;
#endif
  const uint32_t tmem_dF = tmem_base;

  // Roles 0 and 1 run on the whole warp with warp-uniform control flow; one lane issues (see sim_fwd.cu)
  if (warp == 0) {
    // ================= TMA producer: one Y unit (128 rows x C_pad) per stage =================
    Walker wk(args.work);
    Segment sg, nx;
    uint32_t u = 0;
    bool have = wk.next(sg);
    while (have) {
      const bool have_n = wk.next(nx);      // the work item of the next run is fetched while this one streams
      const BwdDev& p = args.p[sg.owner];
      for (int ct = sg.c_begin; ct < sg.c_end; ++ct, ++u) {
        const uint32_t st = u % kBwdStages, ph = (u / kBwdStages) & 1;
        ptx::mbar_wait(&b_empty[st], ph ^ 1, 202);
        if (ptx::elect_one()) {
          ptx::mbar_expect_tx(&b_full[st], KB * kBlkBytes);
          for (int kb = 0; kb < KB; ++kb)
            ptx::tma_load_2d(smB + (size_t)(st * KB + kb) * kBlkBytes, &args.maps[p.y_map], &b_full[st], kb * kKBlk,
                             ct * kTileN);
        }
        __syncwarp();
      }
      sg = nx; have = have_n;
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    constexpr uint32_t idesc_s = ptx::umma_idesc_bf16(128, kBwdSub, 0, 0);  // S  = X Y^T   (B K-major)
    constexpr uint32_t idesc_d = ptx::umma_idesc_bf16(128, CP, 0, 1);       // dX += W Y    (B MN-major)
    const uint32_t b_addr = ptx::smem_u32(smB);
    // descriptor bases of the Y ring: K-major use (S MMAs) and MN-major use (dX MMAs, LBO = next 64-channel block)
    const uint64_t kdesc = ptx::umma_desc_sw128(b_addr, 16, 1024), mdesc = ptx::umma_desc_sw128(b_addr, kBlkBytes, 1024);
    const uint32_t k_lo = (uint32_t)kdesc, k_hi = (uint32_t)(kdesc >> 32);
    const uint32_t m_lo = (uint32_t)mdesc, m_hi = (uint32_t)(mdesc >> 32);
    Walker wk(args.work);
    Segment sg, nx;
    uint32_t t2 = 0, u = 0, seg = 0;         // tiles, units, runs issued so far
    // The tensor pipe buffers only a few MMAs and an S MMA (N = 64) lasts 32 cycles, so scalar code between two
    // MMA groups is a pipe bubble (measured: ~270 of 1300 cycles per tile with one elect block per group).  A tile
    // step therefore does all barrier work first and then issues S(cur+1) and dX(cur) from ONE elect block; the
    // descriptor of a tile is stepped with one 32-bit add per MMA (ptx.cuh:umma_ts2).
    // (called by the elected lane only)
    auto emit_s = [&](uint32_t cur_, uint32_t unit_, uint32_t h_) {
      const uint32_t sb_ = cur_ & 1, st_ = unit_ % kBwdStages;
      const uint32_t lo0 = k_lo + ((st_ * (KB * kBlkBytes) + h_ * (kBwdSub * 128)) >> 4);
      const uint32_t d_tm = tmem_base + kTmS + sb_ * kBwdSub, a_tm = tmem_base + kTmX;
      // S buffer `sb_` also holds W of tile cur_-2: its consumer (the dX MMAs of tile cur_-2) was issued
      // before this point and tcgen05.mma executes in issue order, so no extra barrier is needed
#pragma unroll
      for (int kk = 0; kk < 4 * KB; ++kk)
        ptx::umma_ts2(d_tm, a_tm + kk * 8, lo0 + (((kk >> 2) * kBlkBytes + (kk & 3) * 32) >> 4), k_hi, idesc_s, kk != 0);
      ptx::umma_commit(&s_full[sb_]);
    };
    // W of tile column quarter q lives in columns [16q, 16q+8) of S buffer sb (two bf16 per TMEM column): that is
    // the K = 16 slice q.  Y rows 64h + 16q .. +15 are the matching K slice of B; LBO = next 64-channel block.
    auto emit_d = [&](uint32_t cur_, uint32_t unit_, uint32_t h_, uint32_t first) {
      const uint32_t sb_ = cur_ & 1, st_ = unit_ % kBwdStages;
      const uint32_t lo1 = m_lo + ((st_ * (KB * kBlkBytes) + h_ * (kBwdSub * 128)) >> 4);
      const uint32_t w_tm = tmem_base + kTmS + sb_ * kBwdSub;
#pragma unroll
      for (int q = 0; q < 4; ++q)
        ptx::umma_ts2(tmem_dF, w_tm + q * 16, lo1 + ((q * 16 * 128) >> 4), m_hi, idesc_d, (first != 0) | (q != 0));
      if (h_ == 1) ptx::umma_commit(&b_empty[st_]);
    };
    bool have = wk.next(sg);
    while (have) {
      const bool have_n = wk.next(nx);
      ptx::mbar_wait(x_full, seg & 1, 212);
      ptx::mbar_wait(&b_full[u % kBwdStages], (u / kBwdStages) & 1, 211);
      ptx::tc_fence_after();
      MSCS_TRACE_EV(3, 0, seg);
      const uint32_t ntiles = 2 * (uint32_t)(sg.c_end - sg.c_begin);
#ifdef MSCS_TRACE
      if (blockIdx.x == 5 && lane == 0 && seg < 256u) ptx::g_trace[3 * 2048 + seg * 8 + 2] = ntiles;
      if (blockIdx.x == 5 && lane == 0 && seg == 0) ptx::g_trace[3 * 2048 + 255 * 8 + 7] = (unsigned long long)prof_c0;
#endif
      if (ptx::elect_one()) emit_s(t2, u, 0);
      __syncwarp();
      // the previous run's dX must have been read out before the first dX MMA of this run overwrites it
      ptx::mbar_wait(df_empty, (seg & 1) ^ 1, 213);
      for (uint32_t j = 0; j < ntiles; ++j) {
        const uint32_t cur = t2 + j, sb = cur & 1, unit = u + (j >> 1), h = j & 1;
        const bool has_next = j + 1 < ntiles;
        const uint32_t unit_n = u + ((j + 1) >> 1), h_n = (j + 1) & 1;
        // Issue order S(cur+1) | dX(cur): the S chain of the next tile runs while the epilogue turns S(cur) into W(cur).
        // W(cur) becomes ready about when the S group has been accepted by the pipe, which then holds only a few
        // 32-cycle MMAs: the elected lane waits for the barrier ITSELF and issues dX(cur) at once (re-converging the
        // warp and electing again in between cost ~200 cycles = a pipe bubble on every tile).
        if (ptx::elect_one()) {
          if (has_next) {
            if (h_n == 0) {      // first tile of the next unit: its Y data (requested two units ago)
              ptx::mbar_wait(&b_full[unit_n % kBwdStages], (unit_n / kBwdStages) & 1, 211);
              ptx::tc_fence_after();
            }
            emit_s(cur + 1, unit_n, h_n);
          }
          MSCS_TRACE_EV(0, 0, cur);
          ptx::mbar_spin_wait(&w_full[sb], (cur >> 1) & 1, 214);
          ptx::tc_fence_after();
          MSCS_TRACE_EV(0, 1, cur);
          emit_d(cur, unit, h, j);
        }
        __syncwarp();
        MSCS_TRACE_EV(0, 2, cur);
      }
      if (ptx::elect_one()) ptx::umma_commit(df_full);
      __syncwarp();
      MSCS_TRACE_EV(3, 1, seg);
      t2 += ntiles; u += ntiles >> 1; ++seg;
      sg = nx; have = have_n;
    }
  } else if (warp >= 4) {
    // ================= epilogue: thread = (row, 16-column quarter of a tile) =================
    const int cq = (warp - 4) >> 2, quad = warp & 3;
    const int r_loc = quad * 32 + lane;                     // row inside the block = TMEM lane
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    float* my_cs = cstat + (warp - 4) * (2 * 3 * 32);       // this warp's [2 buffers][cs, cpn, neg][2 tiles x 16 columns]
    const float gout = *args.grad_out;
    Walker wk(args.work);
    Segment sg, nx;
    uint32_t t2 = 0, un = 0, seg = 0;
    bool have = wk.next(sg);
    while (have) {
      const bool have_n = wk.next(nx);      // next run's work item: its dependent global loads overlap this run
      const BwdDev& p = args.p[sg.owner];
      const int row = sg.rb * 128 + r_loc;
      int dev_rows = 0, dev_cols = 0;
      if constexpr (DEV) { dev_rows = *args.rows_dev[sg.owner]; dev_cols = *args.cols_dev[sg.owner]; }
      if (warp == 4) MSCS_TRACE_EV(3, 3, 64u + seg);
      // ---- X rows of this run -> TMEM (A operand layout: lane = row, two bf16 per column).  Every S MMA of the
      // previous run has completed: this warp has passed the s_full wait of its last tile.
      if (cq < KB) {
        const uint4* src = reinterpret_cast<const uint4*>(p.x_rows + (size_t)row * CP + cq * 64);   // rows are padded
        uint32_t xv[32];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const uint4 q4 = __ldg(src + i);
          xv[4 * i] = q4.x; xv[4 * i + 1] = q4.y; xv[4 * i + 2] = q4.z; xv[4 * i + 3] = q4.w;
        }
        ptx::tmem_st32(tmem_base + lane_base + kTmX + cq * 32, xv);
        ptx::tmem_st_wait();
      }
      if (warp == 4) MSCS_TRACE_EV(3, 4, 64u + seg);
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(x_full);
      const bool valid = row < (DEV ? dev_rows : p.n_rows);
      int p0 = 0, p1 = 0;
      if (valid) { const int y = p.row_cls[row]; p0 = p.col_seg[y]; p1 = p.col_seg[y + 1]; }
      const unsigned plen = (unsigned)(p1 - p0);
      int wmin = valid ? p0 : 0x7fffffff, wmax = valid ? p1 : 0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        wmin = min(wmin, __shfl_xor_sync(0xffffffffu, wmin, o));
        wmax = max(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
      }
      const float rcs = (valid && p.row_cs) ? p.row_cs[row] : 0.f;
      const float rcpn = (valid && p.row_cpn) ? p.row_cpn[row] : 0.f;
      const float rneg = (valid && p.row_neg) ? p.row_neg[row] : 1.f;
      const int self_col = p.self_mask ? row : -1;
      const float scale = p.scale_log2;
      const uint64_t scale2 = ptx::pack2(scale, scale), rcs2 = ptx::pack2(rcs, rcs);
      // column coefficients: lane l fetches those of column 16 cq + (l & 15) of tile (l >> 4) of the NEXT unit
      // (parked in registers), then the warp stages them in its own smem slot -- no cross-warp synchronisation
      float pf_s = 0.f, pf_pn = 0.f, pf_neg = 1.f;
      auto prefetch_cols = [&](int ct_) {
        pf_s = 0.f; pf_pn = 0.f; pf_neg = 1.f;
        if (ct_ < sg.c_end) {
          const int c = ct_ * kTileN + (lane >> 4) * kBwdSub + cq * 16 + (lane & 15);
          if (c < (DEV ? dev_cols : p.n_cols)) {
            if (p.col_cs) pf_s = p.col_cs[c];
            if (p.col_cpn) pf_pn = p.col_cpn[c];
            if (p.col_neg) pf_neg = p.col_neg[c];
          }
        }
      };
      auto publish_cols = [&](uint32_t b_) {
        float* cs = my_cs + b_ * 96;
        cs[lane] = pf_s; cs[32 + lane] = pf_pn; cs[64 + lane] = pf_neg;
        __syncwarp();
      };
      prefetch_cols(sg.c_begin);
      publish_cols(un & 1);
      if (warp == 4) MSCS_TRACE_EV(3, 5, 64u + seg);
      for (int ct = sg.c_begin; ct < sg.c_end; ++ct, ++un) {
        const float* cs_unit = my_cs + (un & 1) * 96;
        prefetch_cols(ct + 1);
#pragma unroll
        for (int h = 0; h < 2; ++h, ++t2) {
          const uint32_t sb = t2 & 1;
          const int cb = ct * kTileN + h * kBwdSub + cq * 16;      // first global column of this thread's quarter
          const float* cs_s = cs_unit + h * 16; const float* cs_pn = cs_s + 32; const float* cs_neg = cs_s + 64;
          const bool touches = !(cb + 16 <= wmin || cb >= wmax);
          // (Polling instead -- all 16 warps with test_wait, or one warp per SM sub-partition with the other three
          // parked in a named barrier -- measured no faster than the suspending try_wait.)
          ptx::mbar_wait(&s_full[sb], (t2 >> 1) & 1, 221);
          ptx::tc_fence_after();
          const uint32_t taddr = tmem_base + lane_base + kTmS + sb * kBwdSub + cq * 16;
          uint32_t v[16];
          ptx::tmem_ld16(taddr, v);
          ptx::tmem_ld_wait16(v);
          uint32_t packed[8];
          if (!touches) {
            // W = exp2(S scale) (cS_row + cS_col), two columns per packed fp32x2 instruction
#pragma unroll
            for (int c = 0; c < 16; c += 4) {
              const float4 cc = *reinterpret_cast<const float4*>(cs_s + c);
#pragma unroll
              for (int q = 0; q < 2; ++q) {
                // (MUFU only: a degree-3 polynomial on the FMA pipe for every second pair measured slower -- the FMA
                // pipe becomes the bound)
                float x0, x1;
                ptx::unpack2(ptx::mul2(ptx::pack2u(v[c + 2 * q], v[c + 2 * q + 1]), scale2), x0, x1);
                const uint64_t e2 = ptx::pack2(ptx::ex2(x0), ptx::ex2(x1));
                const uint64_t c2 = ptx::add2(rcs2, q == 0 ? ptx::pack2(cc.x, cc.y) : ptx::pack2(cc.z, cc.w));
                float w0, w1;
                ptx::unpack2(ptx::mul2(e2, c2), w0, w1);
                packed[(c >> 1) + q] = pack_bf16(w0, w1);
              }
            }
          } else {
#pragma unroll
            for (int c = 0; c < 16; c += 2) {
              float w[2];
#pragma unroll
              for (int q = 0; q < 2; ++q) {
                const int j = c + q;
                const int col = cb + j;
                const float e = ptx::ex2(__uint_as_float(v[j]) * scale);
                const bool ispos = (unsigned)(col - p0) < plen;
                const float wn = e * (rcs + cs_s[j]);
                const float wp = -(rcpn * ptx::rcp(e + rneg) + cs_pn[j] * ptx::rcp(e + cs_neg[j]));
                w[q] = ispos ? (col == self_col ? 0.f : wp) : wn;
              }
              packed[c >> 1] = pack_bf16(w[0], w[1]);
            }
          }
          // 16 logits -> 8 packed columns, written over S columns this thread has already read
          ptx::tmem_st8(taddr, packed);
          ptx::tmem_st_wait();
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&w_full[sb]);
          MSCS_TRACE_EV(1 + ((warp - 4) >> 3), (warp - 4) & 7, t2);      // arrival time of each epilogue warp
        }
        publish_cols((un & 1) ^ 1);      // every lane is past its reads of that slot (the __syncwarp above)
      }
      // ---- flush dX: this warp drains channel quarter cq of its 32 rows (the next run's data is requested first) ----
      if (warp == 4) MSCS_TRACE_EV(3, 0, 64u + seg);
      if (have_n && cq < KB)      // warm L2 with the next run's X rows while this run is flushed
        asm volatile("prefetch.global.L2 [%0];" ::"l"(args.p[nx.owner].x_rows + (size_t)(nx.rb * 128 + r_loc) * CP + cq * 64));
      ptx::mbar_wait(df_full, seg & 1, 222);
      ptx::tc_fence_after();
      if (warp == 4) MSCS_TRACE_EV(3, 1, 64u + seg);
      const float sc = p.out_scale * gout;
      float* drow = p.dF + (size_t)row * p.ld;
#pragma unroll 1
      for (int c0 = cq * (CP / 4); c0 < (cq + 1) * (CP / 4); c0 += 16) {
        uint32_t uu[16];
        ptx::tmem_ld16(tmem_dF + lane_base + c0, uu);
        ptx::tmem_ld_wait16(uu);
        if (valid) {
#pragma unroll
          for (int c = 0; c < 16; c += 4)
            red_add_v4(drow + c0 + c, __uint_as_float(uu[c]) * sc, __uint_as_float(uu[c + 1]) * sc,
                       __uint_as_float(uu[c + 2]) * sc, __uint_as_float(uu[c + 3]) * sc);
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(df_empty);
      if (warp == 4) MSCS_TRACE_EV(3, 2, 64u + seg);
      ++seg;
      sg = nx; have = have_n;
    }
  }
  __syncwarp();
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) ptx::tmem_dealloc(tmem_base, 512);
#ifdef MSCS_TRACE
  if (blockIdx.x == 5 && threadIdx.x == 0) ptx::g_trace[3 * 2048 + 255 * 8 + 6] = (unsigned long long)clock64();
  if (threadIdx.x == 0 && blockIdx.x < 256) {      // per-CTA duration and start offset (globaltimer ns)
    ptx::g_trace[3 * 2048 + 1024 + blockIdx.x] = (unsigned long long)(clock64() - prof_c0);
    ptx::g_trace[3 * 2048 + 1280 + blockIdx.x] = prof_t0;
    ptx::g_trace[3 * 2048 + 1536 + blockIdx.x] = ptx::globaltimer_ns();
  }
#endif
#ifdef MSCS_WAIT_PROFILE
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    atomicAdd(&ptx::g_wait_ns[31], ptx::globaltimer_ns() - prof_t0);
    atomicAdd(&ptx::g_wait_cnt[31], (unsigned long long)(clock64() - prof_c0));
  }
#endif
}

}  // namespace mscs

using namespace mscs;

template <int KB, bool DEV>
static int launch_bwd(const BwdArgs& args, cudaStream_t st) {
  const size_t smem = bwd_smem_bytes(KB);
  if (int rc = ensure_trap_buffer()) return rc;
  MSCS_CUDA(cudaFuncSetAttribute(k_sim_bwd<KB, DEV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  MSCS_CUDA(launch_k(k_sim_bwd<KB, DEV>, persistent_ctas(), kBwdThreads, smem, st, args));
  MSCS_LAUNCH_CHECK();
  return 0;
}

extern "C" int mscs_sim_backward(const mscs_sim_job* job, const float* grad_out, float* const* dF_sets,
                                 const int32_t* dF_ld, void* stream_) {
  return mscs_sim_backward_sets(job, grad_out, dF_sets, dF_ld, 0xffffffffu, stream_);
}

// Only the passes whose ROW set is in `set_mask` (bit s = anchor set s): the pooled mode launches the backward
// set by set so that the exchange of one set's gradient rows overlaps the tensor work of the next.
extern "C" int mscs_sim_backward_sets(const mscs_sim_job* job, const float* grad_out, float* const* dF_sets,
                                      const int32_t* dF_ld, uint32_t set_mask, void* stream_) {
  int rc = validate_job(job);
  if (rc) return rc;
  MSCS_CHECK_ARG(job->work && grad_out && dF_sets && dF_ld, "null pointer argument");
  // device-resident row counts (n1_dev / n2_dev): for every term or for none; N1 / N2 are then upper bounds that size
  // the work table and the tensor maps, and the kernels read the actual counts
  const bool dev_counts = job->terms[0].n1_dev != nullptr;
  for (int t = 0; t < job->num_terms; ++t)
    MSCS_CHECK_ARG((job->terms[t].n1_dev != nullptr) == dev_counts && (job->terms[t].n2_dev != nullptr) == dev_counts,
                   "term %d: n1_dev / n2_dev must be set for every term or for none", t);
  cudaStream_t st = (cudaStream_t)stream_;
  BwdPass passes[MSCS_MAX_PASSES];
  int np = build_passes(job, passes);
  {
    int kept = 0;
    for (int i = 0; i < np; ++i)
      if ((set_mask >> passes[i].row_set) & 1u) passes[kept++] = passes[i];
    np = kept;
    if (np == 0) return 0;
  }
  // the backward work tables live after the two forward tables in job->work
  size_t fwd_items = 0, ranges = 0;
  for (int t = 0; t < job->num_terms; ++t) {
    fwd_items += (size_t)ceil_div(job->terms[t].N2, 256);
    ranges += align_up(sizeof(int2) * (size_t)job->terms[t].N1, 64) +
              align_up(sizeof(int2) * (size_t)ceil_div(job->terms[t].N1, 128) * 4, 64);
  }
  char* w = (char*)job->work + 4096 + ranges +
            2 * (align_up(sizeof(WorkItem) * fwd_items, 64) + align_up(sizeof(int) * (fwd_items + 1), 64));
  BwdArgs args{};
  args.grad_out = grad_out;
  const void* bases[MSCS_MAX_SCALES]; int nmaps = 0;
  auto map_of = [&](const void* base, int rows) -> int {
    for (int i = 0; i < nmaps; ++i) if (bases[i] == base) return i;
    if (nmaps == MSCS_MAX_SCALES) return -1;
    if (make_tensor_map(&args.maps[nmaps], base, (rows + 255) / 256 * 256, job->C_pad)) return -2;
    bases[nmaps] = base;
    return nmaps++;
  };
  BuildArgs b{};
  int nitems = 0;
  for (int i = 0; i < np; ++i) {
    const BwdPass& p = passes[i];
    const int ym = map_of(p.y_bf16, p.n_cols);
    if (ym == -2) return -1;
    MSCS_CHECK_ARG(ym >= 0, "too many distinct operand matrices");
    MSCS_CHECK_ARG(dF_sets[p.row_set] && dF_ld[p.row_set] >= job->C_pad && dF_ld[p.row_set] % 4 == 0,
                   "pass %d: dF buffer of set %d missing or leading dimension < C_pad", i, p.row_set);
    args.p[i] = BwdDev{p.row_cls, p.col_seg, p.row_cs, p.row_cpn, p.row_neg, p.col_cs, p.col_cpn, p.col_neg,
                       (const __nv_bfloat16*)p.x_bf16, dF_sets[p.row_set], dF_ld[p.row_set], p.n_rows, p.n_cols,
                       p.self_mask, ym, p.scale_log2, p.out_scale};
    b.t[i] = BuildTerm{p.row_cls, p.col_seg, p.n_rows, p.n_cols, nitems, p.rb_lo, 0, 1 << 30, p.n_rows_dev, p.n_cols_dev};
    args.rows_dev[i] = p.n_rows_dev; args.cols_dev[i] = p.n_cols_dev;
    nitems += p.rb_hi - p.rb_lo;
  }
  b.num_terms = np; b.nitems = nitems; b.rows_per_item = 128; b.mode = 0;
  b.pad = 6;      // a run start costs about as much as 6 units (X load, pipeline fill, dX flush: ~15k cycles)
  static const int pad_env = [] { const char* e = getenv("MSCS_BWD_PAD"); return e ? atoi(e) : -1; }();
  if (pad_env >= 0) b.pad = pad_env;
  b.items = (WorkItem*)w; w += align_up(sizeof(WorkItem) * (size_t)nitems, 64);
  b.prefix = (int*)w;
  rc = launch_build_work(b, st);
  if (rc) return rc;
  args.work = WorkTable{b.items, b.prefix, nitems, b.pad};
  if (dev_counts) {
    switch (job->C_pad / 64) {
      case 1: return launch_bwd<1, true>(args, st);
      case 2: return launch_bwd<2, true>(args, st);
      case 3: return launch_bwd<3, true>(args, st);
      default: return launch_bwd<4, true>(args, st);
    }
  }
  switch (job->C_pad / 64) {
    case 1: return launch_bwd<1, false>(args, st);
    case 2: return launch_bwd<2, false>(args, st);
    case 3: return launch_bwd<3, false>(args, st);
    default: return launch_bwd<4, false>(args, st);
  }
}

// debug: read and reset the barrier wait profile of this translation unit (ns and count per tag % 32)
extern "C" int mscs_debug_wait_profile_bwd(unsigned long long* ns_out, unsigned long long* cnt_out) {
  MSCS_CUDA(cudaDeviceSynchronize());
  MSCS_CUDA(cudaMemcpyFromSymbol(ns_out, ptx::g_wait_ns, sizeof(unsigned long long) * 32));
  MSCS_CUDA(cudaMemcpyFromSymbol(cnt_out, ptx::g_wait_cnt, sizeof(unsigned long long) * 32));
  unsigned long long zero[32] = {};
  MSCS_CUDA(cudaMemcpyToSymbol(ptx::g_wait_ns, zero, sizeof(zero)));
  MSCS_CUDA(cudaMemcpyToSymbol(ptx::g_wait_cnt, zero, sizeof(zero)));
  return 0;
}

// debug (trace build only): copy out and reset the event trace of the backward kernel; returns the event count
extern "C" int mscs_debug_trace_bwd(unsigned long long* out, int max_events) {
#ifdef MSCS_TRACE
  MSCS_CUDA(cudaDeviceSynchronize());
  const int n = max_events < 8192 ? max_events : 8192;
  MSCS_CUDA(cudaMemcpyFromSymbol(out, ptx::g_trace, sizeof(unsigned long long) * n));
  static unsigned long long zeros[8192];
  MSCS_CUDA(cudaMemcpyToSymbol(ptx::g_trace, zeros, sizeof(zeros)));
  return n;
#else
  (void)out; (void)max_events;
  return 0;
#endif
}
