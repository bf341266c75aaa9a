// sim_fwd.cu -- K3: fused similarity + loss forward on tcgen05 / TMEM, TMA-fed.
//
// Replaces, for every term of a call at once (V2.py:127-192, _ms.py:84-161):
//   normalised anchors x keys^T / tau, the positive / negative masks, exp, the row sums and the
//   per-pair log-probabilities -- without ever materialising the N1 x N2 logits.
// Two sweeps of the same kernel (the positive terms need the complete negative sums):
//   MODE 0  all tiles:               neg_i  = sum_{y_j != y_i} exp(l_ij)
//   MODE 1  class-diagonal tiles:    pos_i  = sum_{j in P_i} [l_ij - log(exp(l_ij) + neg_i)],
//                                    S_i    = sum_{j in P_i} 1/(exp(l_ij) + neg_i)
//
// CTA = a block of 256 KEYS resident in smem (the N = 256 operand of the MMA) x a run of 128-ANCHOR
// tiles streamed through a TMA ring (the M = 128 operand).  One 128x256x16 MMA per K step: the
// shared-memory operand traffic per FLOP is 25% lower than with 128x128 MMAs (which measured at
// ~45% of the tensor peak here, shared-memory bound) and the accumulate dependency is hidden.
// Accumulators (128 lanes x 256 columns) are double-buffered in TMEM.
// Warp roles: 0 TMA producer, 1 MMA issuer, 2 TMEM allocator, 4..11 / 12..19 epilogue groups 0 / 1
// (even / odd tiles): thread = (anchor row of the tile, 128-key half); partial row sums go out with
// one atomicAdd per row, half and tile.
#include "sim_tc.cuh"
#include <stdlib.h>
#ifdef MSCS_TRACE      // the forward trace records ONE sweep (the other would overwrite it): -DMSCS_TRACE_MODE=0|1
#ifndef MSCS_TRACE_MODE
#define MSCS_TRACE_MODE 0
#endif
#undef MSCS_TRACE_EV
#define MSCS_TRACE_EV(slot, k, tile)                                                                 \
  do {                                                                                               \
    if (MODE == MSCS_TRACE_MODE && blockIdx.x == 5 && (threadIdx.x & 31) == 0 && (tile) < 256u)                    \
      mscs::ptx::g_trace[(slot) * 2048 + (tile) * 8 + (k)] = (unsigned long long)clock64();          \
  } while (0)
#endif

namespace mscs {

constexpr int kFwdKeys = 256;       // resident key block = N of the MMA
// Two epilogue groups of 8 warps: group g owns accumulator buffer g, i.e. every second tile, so the TMEM-load
// latency and barrier hand-over of one tile overlap the exponentials of the other (with one group the
// MUFU unit idled half of the time although it is the busiest unit of the pass).
// Round-2 event traces (tools/trace_fwd.py, profiles/r02_fwd_trace.md) of this and four alternative epilogue
// structures: here a tile takes ~2900 cycles against 2048 of MMA time (MMA 1900 + completion lag 500 + exponentials
// ~3200 of one group with the MUFU shared by both, per buffer).  All sixteen warps on every tile with the accumulator
// copied to registers and released before the math (held ~500 cycles): 3200-3800 per tile -- the warps then run their
// non-MUFU phases in lock step; the same software-pipelined over tiles: 5200; with masks fetched only on
// class-diagonal tiles: 3100; phase-staggered start: no change.  The ping-pong groups stay.
constexpr int kFwdEpiWarps = 16;
constexpr int kFwdThreads = 128 + 32 * kFwdEpiWarps;
constexpr int kFwdColsPerThread = kFwdKeys / 2;      // thread = (anchor row, 128-key half) of its group's tiles
constexpr int kFwdStages = 5;
// (Tried in round 2: accumulating the 128 x 256 tile as two 128-column halves with N = 128 MMAs and one full / empty
// barrier pair per half -- four accumulators in flight, the first half's warps start 1000 cycles earlier.  Correct, but
// the forward stage went from 0.223 to 0.393 ms at cfg-2: the N = 128 form reads the anchor K-blocks twice and runs at
// the shared-memory read limit of the MMA unit (128 B/clk) next to the TMA writes.  profiles/r02_fwd_trace.md.)
constexpr int kAccBars = 2;

struct FwdTerm {
  const int* a_cls; const int* k_seg;
  const int2* row_range;   // per anchor row: [first, last+1) positive key rows   (k_row_ranges)
  const int2* grp_range;   // per group of 32 anchor rows: union of the above
  float* neg; float* pos; float* ssum;
  int N1, N2, self_mask, a_map, k_map;
  float scale_log2;
  const int* n1_dev; const int* n2_dev;      // optional device-resident row counts (N1 / N2 are then upper bounds)
};
struct FwdArgs {
  alignas(64) CUtensorMap maps[MSCS_MAX_SCALES];
  FwdTerm t[MSCS_MAX_TERMS];
  WorkTable work;
};

__host__ __device__ constexpr size_t fwd_smem_bytes(int KB) {
  return 1024 /*alignment slack*/ + (size_t)(2 * KB + kFwdStages) * kBlkBytes + 256 /*barriers*/;
}

// 16 unmasked logits -> partial sums of exp2(v * scale), TWO elements per instruction wherever the pipe allows it
// (packed fp32x2 multiply / add; MUFU.EX2 itself is scalar).  Per pair: FMUL2 + 2 MUFU + FADD2.  (Moving a share of
// the exponentials to a polynomial on the FMA pipe measured no faster, DESIGN.md §4.)
__device__ __forceinline__ void fast_chunk(const uint32_t (&cur)[16], uint64_t scale2, uint64_t& acc_a, uint64_t& acc_b) {
#pragma unroll
  for (int c = 0; c < 16; c += 2) {
    float x0, x1;
    ptx::unpack2(ptx::mul2(ptx::pack2u(cur[c], cur[c + 1]), scale2), x0, x1);
    const uint64_t e2 = ptx::pack2(ptx::ex2(x0), ptx::ex2(x1));
    if (c & 2) acc_b = ptx::add2(acc_b, e2); else acc_a = ptx::add2(acc_a, e2);
  }
}

// one 16-column chunk of the negative sweep: unmasked when no row of this warp has a positive in it (and it lies
// inside the key set), otherwise per-element masks.  (16 columns: two chunks in flight cost 32 registers, which
// leaves the compiler room to overlap the MUFU latencies of neighbouring pairs; with 32-column chunks every pair
// went through the same register pair.)
__device__ __forceinline__ void neg_chunk(const uint32_t (&cur)[16], int c0, int tN2, int wmin, int wmax, int p0,
                                          unsigned plen, float scale, uint64_t scale2, uint64_t& acc_a, uint64_t& acc_b,
                                          float& acc_m) {
  const bool fast = (c0 + 16 <= wmin || c0 >= wmax) && (c0 + 16 <= tN2);
  if (fast) {
    fast_chunk(cur, scale2, acc_a, acc_b);
  } else if (c0 < tN2) {
#pragma unroll
    for (int c = 0; c < 16; ++c) {
      const int col = c0 + c;
      const float e = ptx::ex2(__uint_as_float(cur[c]) * scale);
      const bool isneg = ((unsigned)(col - p0) >= plen) && (col < tN2);
      acc_m += isneg ? e : 0.f;
    }
  }
}

#ifdef MSCS_WAIT_PROFILE
// per CTA and sweep of the last launch: start / end (globaltimer ns), SM cycles, SM id  (profiling build only)
static __device__ unsigned long long g_cta_span[2][160][4];
#endif

template <int KB, int MODE>
__global__ void __launch_bounds__(kFwdThreads, 1) k_sim_fwd(const __grid_constant__ FwdArgs args) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smK = smem;                                   // resident keys  [KB][256 rows][128 B]
  uint8_t* smA = smem + (size_t)2 * KB * kBlkBytes;      // anchor ring    [stages][128 rows][128 B]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smA + (size_t)kFwdStages * kBlkBytes);
  uint64_t* a_full = bars;                    // [stages]  streamed anchor K-blocks
  uint64_t* a_empty = bars + kFwdStages;      // [stages]
  uint64_t* k_full = bars + 2 * kFwdStages;   // resident key block
  uint64_t* k_empty = k_full + 1;
  uint64_t* acc_full = k_full + 2;            // [kAccBars]
  uint64_t* acc_empty = acc_full + kAccBars;  // [kAccBars]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + kAccBars);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  pdl_trigger();
  if (warp == 0 && lane == 0) {
    for (int i = 0; i < kFwdStages; ++i) { ptx::mbar_init(&a_full[i], 1); ptx::mbar_init(&a_empty[i], 1); }
    ptx::mbar_init(k_full, 1); ptx::mbar_init(k_empty, 1);
    for (int i = 0; i < kAccBars; ++i) { ptx::mbar_init(&acc_full[i], 1); ptx::mbar_init(&acc_empty[i], kFwdEpiWarps / kAccBars); }
    ptx::fence_barrier_init();
  }
  if (warp == 2) ptx::tmem_alloc(tmem_slot, 512);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
#ifdef MSCS_TRACE
  if (MODE == MSCS_TRACE_MODE && blockIdx.x == 5 && threadIdx.x == 0) ptx::g_trace[3 * 2048 + 255 * 8 + 5] = (unsigned long long)clock64();
#endif
  pdl_wait();       // barriers and tensor memory are set up while the previous grid drains
#ifdef MSCS_TRACE
  if (MODE == MSCS_TRACE_MODE && blockIdx.x == 5 && threadIdx.x == 0) ptx::g_trace[3 * 2048 + 255 * 8 + 7] = (unsigned long long)clock64();
#endif
#ifdef MSCS_WAIT_PROFILE     // effective SM clock of this launch: slot 31 accumulates (ns, cycles) of CTA 0
  const unsigned long long prof_t0 = ptx::globaltimer_ns();
  const long long prof_c0 = clock64();
#endif

  // Roles 0 and 1 are executed by the WHOLE warp (waits, loop control and descriptor arithmetic stay
  // warp-uniform); only the TMA / MMA instructions themselves are issued by one elected lane.
  if (warp == 0) {
    // ================= TMA producer =================
    Walker wk(args.work);
    Segment sg;
    int stage = 0; uint32_t phase = 0, k_phase = 0;
    while (wk.next(sg)) {
      const FwdTerm& t = args.t[sg.owner];
      ptx::mbar_wait(k_empty, k_phase ^ 1, 101);
      if (ptx::elect_one()) {
        ptx::mbar_expect_tx(k_full, 2 * KB * kBlkBytes);
        for (int kb = 0; kb < KB; ++kb)
          for (int h = 0; h < 2; ++h)
            ptx::tma_load_2d(smK + (size_t)(kb * 2 + h) * kBlkBytes, &args.maps[t.k_map], k_full, kb * kKBlk,
                             sg.rb * kFwdKeys + h * 128);
      }
      k_phase ^= 1;
      for (int rt = sg.c_begin; rt < sg.c_end; ++rt)
        for (int kb = 0; kb < KB; ++kb) {
          ptx::mbar_wait(&a_empty[stage], phase ^ 1, 102);
          if (ptx::elect_one()) {
            ptx::mbar_expect_tx(&a_full[stage], kBlkBytes);
            ptx::tma_load_2d(smA + (size_t)stage * kBlkBytes, &args.maps[t.a_map], &a_full[stage], kb * kKBlk,
                             rt * 128);
          }
          if (++stage == kFwdStages) { stage = 0; phase ^= 1; }
        }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    constexpr uint32_t idesc = ptx::umma_idesc_bf16(128, kFwdKeys, 0, 0);
    Walker wk(args.work);
    Segment sg;
    int stage = 0; uint32_t phase = 0, k_phase = 0, it = 0;
    const uint32_t k_addr = ptx::smem_u32(smK), a_addr = ptx::smem_u32(smA);
    while (wk.next(sg)) {
      MSCS_TRACE_EV(0, 3, it);
      ptx::mbar_wait(k_full, k_phase, 111); k_phase ^= 1;
      ptx::tc_fence_after();
      MSCS_TRACE_EV(0, 4, it);
      for (int rt = sg.c_begin; rt < sg.c_end; ++rt, ++it) {
        const uint32_t buf = it & 1;
        MSCS_TRACE_EV(0, 0, it);
        ptx::mbar_wait(&acc_empty[buf], ((it >> 1) & 1) ^ 1, 112);
        ptx::tc_fence_after();
        MSCS_TRACE_EV(0, 1, it);
        for (int kb = 0; kb < KB; ++kb) {
          ptx::mbar_wait(&a_full[stage], phase, 113);
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint64_t ad = ptx::umma_desc_sw128(a_addr + stage * kBlkBytes + k * 32, 16, 1024);
              const uint64_t bd = ptx::umma_desc_sw128(k_addr + kb * 2 * kBlkBytes + k * 32, 16, 1024);
              ptx::umma_ss(tmem_base + buf * kFwdKeys, ad, bd, idesc, (kb | k) != 0);
            }
            ptx::umma_commit(&a_empty[stage]);
          }
          __syncwarp();
          if (++stage == kFwdStages) { stage = 0; phase ^= 1; }
        }
        if (ptx::elect_one()) ptx::umma_commit(&acc_full[buf]);
        __syncwarp();
        MSCS_TRACE_EV(0, 2, it);
      }
      if (ptx::elect_one()) ptx::umma_commit(k_empty);
      __syncwarp();
    }
  } else if (warp >= 4) {
    // ================= epilogue: thread = (anchor row of the tile, 128-key half) =================
    constexpr int CPT = kFwdColsPerThread, NCH = CPT / 32;
    const int grp = (warp - 4) >> 3, ch = ((warp - 4) >> 2) & 1, quad = warp & 3;
    Walker wk(args.work);
    Segment sg;
    uint32_t it = 0;
    while (wk.next(sg)) {
      const FwdTerm& t = args.t[sg.owner];
      const int tN1 = t.n1_dev ? *t.n1_dev : t.N1, tN2 = t.n2_dev ? *t.n2_dev : t.N2;
      const int cb = sg.rb * kFwdKeys + ch * CPT;          // first key column of this thread's quarter
      const float scale = t.scale_log2;
      // positive key range of each row (and of its 32-row group) comes precomputed from k_row_ranges; the
      // loads are issued before the accumulator wait (the other group keeps the SM busy meanwhile)
      for (int rt = sg.c_begin; rt < sg.c_end; ++rt, ++it) {
        const uint32_t buf = it & 1;
        if (buf != (uint32_t)grp) continue;
        const int row = rt * 128 + quad * 32 + lane;
        const bool valid = row < tN1;
        const int2 n_gr = t.grp_range[rt * 4 + quad];
        const int2 n_rr = valid ? t.row_range[row] : make_int2(0, 0);
        const float negi = (MODE == 1 && valid) ? t.neg[row] : 1.f;
        const int p0 = n_rr.x, p1 = n_rr.y, wmin = n_gr.x, wmax = n_gr.y;
        const unsigned plen = (unsigned)(p1 - p0);
        const int self_col = t.self_mask ? row : -1;
        const bool touches = !(cb + CPT <= wmin || cb >= wmax);
        float acc0 = 0.f, acc1 = 0.f;   // MODE 0: acc0 = masked-chunk sum; MODE 1: acc0 = pos (log2 units), acc1 = S
        uint64_t acc_a = 0ull, acc_b = 0ull;      // MODE 0: packed partial sums of the unmasked chunks
#ifdef MSCS_TRACE
        const int tslot = warp == 4 ? 1 : (warp == 11 ? 2 : (warp == 12 ? 3 : -1));
        if (tslot > 0) MSCS_TRACE_EV(tslot, 0, it);
#endif
        ptx::mbar_wait(&acc_full[buf], (it >> 1) & 1, 121);
        ptx::tc_fence_after();
#ifdef MSCS_TRACE
        if (tslot > 0) MSCS_TRACE_EV(tslot, 1, it);
#endif
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + buf * kFwdKeys + ch * CPT;
        if (MODE == 0) {
          if (cb < tN2) {      // a half that lies entirely in the zero padding of the key block has no work
            // two chunks per iteration (the register double buffer keeps compile-time indices); rolled: the fully
            // unrolled body missed the instruction cache at the head of every chunk (11 % of the stall samples)
            constexpr int NC16 = CPT / 16;
            static_assert(NC16 % 2 == 0, "two chunks per iteration");
            const uint64_t scale2 = ptx::pack2(scale, scale);
            uint32_t va[16], vb[16];
            ptx::tmem_ld16(taddr, va);
            ptx::tmem_ld_wait16(va);
#pragma unroll 1
            for (int c4 = 0; c4 < NC16; c4 += 2) {
              ptx::tmem_ld16(taddr + (c4 + 1) * 16, vb);
              neg_chunk(va, cb + c4 * 16, tN2, wmin, wmax, p0, plen, scale, scale2, acc_a, acc_b, acc0);
              ptx::tmem_ld_wait16(vb);
              if (c4 + 2 < NC16) ptx::tmem_ld16(taddr + (c4 + 2) * 16, va);
              neg_chunk(vb, cb + (c4 + 1) * 16, tN2, wmin, wmax, p0, plen, scale, scale2, acc_a, acc_b, acc0);
              if (c4 + 2 < NC16) ptx::tmem_ld_wait16(va);
            }
          }
        } else if (touches) {
          // Positive sweep.  The event trace (tools/trace_fwd1.py) showed ~11.7k cycles per tile in this epilogue with
          // three MUFU ops (ex2, lg2, rcp) and ~14 issue slots per element, for 8 % of the tiles 56 us.  With
          // den = e + neg_i and u = e / neg_i:  lg2(den) = lg2(neg_i) + lg2(1 + u),  1/den = (1/neg_i) / (1 + u), and a
          // positive's e is normally a tiny fraction of the row's negative sum (u ~ 1e-4 at cfg-2), so both become
          // short series on the FMA pipe -- ln(1+u) = u - u^2/2 + u^3/3 (error u^4/4), 1/(1+u) = 1 - u + u^2 - u^3
          // (error u^4) -- evaluated two elements per instruction; ONE MUFU op per element is left.  Chunks of 16
          // columns that lie inside the positive range of EVERY row of the warp and off the diagonal need no masks
          // (rows are class-sorted: all but the warps on a class boundary).  Anything else -- mixed chunks, or a chunk
          // where some e reaches neg_i / 64 -- takes the per-element path with lg2 / rcp.
          const float rneg = valid ? ptx::rcp(negi) : 1.f, lneg = valid ? ptx::lg2(negi) : 0.f;
          int fmin = valid ? p0 : 0x7fffffff, fmax = valid ? p1 : 0;      // columns positive for every row of the warp
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            fmin = max(fmin, __shfl_xor_sync(0xffffffffu, fmin, o));
            fmax = min(fmax, __shfl_xor_sync(0xffffffffu, fmax, o));
          }
          const int row0 = rt * 128 + quad * 32;      // diagonal columns of this warp's rows: [row0, row0 + 32)
          const uint64_t scale2 = ptx::pack2(scale, scale), rneg2 = ptx::pack2(rneg, rneg);
          const uint64_t one2 = ptx::pack2(1.f, 1.f), mone2 = ptx::pack2(-1.f, -1.f), mhalf2 = ptx::pack2(-0.5f, -0.5f),
                         third2 = ptx::pack2(0.3333333433f, 0.3333333433f), ml2e2 = ptx::pack2(-kLog2e, -kLog2e);
#pragma unroll 1
          for (int c4 = 0; c4 < CPT / 16; ++c4) {
            const int c0 = cb + c4 * 16;
            if (c0 + 16 <= wmin || c0 >= wmax) continue;      // warp-uniform
            uint32_t v[16];
            ptx::tmem_ld16(taddr + c4 * 16, v);
            ptx::tmem_ld_wait16(v);
            const bool full = c0 >= fmin && c0 + 16 <= fmax && !(t.self_mask && c0 < row0 + 32 && c0 + 16 > row0);
            bool done = false;
            if (full) {      // warp-uniform
              uint64_t plg2 = 0ull, prc2 = 0ull;
              float emax = 0.f;
#pragma unroll
              for (int c = 0; c < 16; c += 2) {
                const uint64_t x2 = ptx::mul2(ptx::pack2u(v[c], v[c + 1]), scale2);      // logits in log2 units
                float x0, x1;
                ptx::unpack2(x2, x0, x1);
                const float e0 = ptx::ex2(x0), e1 = ptx::ex2(x1);
                emax = fmaxf(emax, fmaxf(e0, e1));
                const uint64_t u2 = ptx::mul2(ptx::pack2(e0, e1), rneg2);
                uint64_t l = ptx::fma2(u2, third2, mhalf2);
                l = ptx::mul2(u2, ptx::fma2(u2, l, one2));                               // ln(1 + u)
                uint64_t r = ptx::fma2(u2, mone2, one2);
                r = ptx::fma2(u2, ptx::fma2(u2, r, mone2), one2);                        // 1 / (1 + u)
                plg2 = ptx::add2(plg2, ptx::fma2(l, ml2e2, x2));                         // x - lg2(1 + u)
                prc2 = ptx::add2(prc2, r);
              }
              if (!__any_sync(0xffffffffu, emax * rneg >= 0.015625f)) {
                float a0, a1, b0, b1;
                ptx::unpack2(plg2, a0, a1); ptx::unpack2(prc2, b0, b1);
                acc0 += fmaf(-16.f, lneg, a0 + a1);
                acc1 = fmaf(b0 + b1, rneg, acc1);
                done = true;
              }
            }
            if (!done) {
#pragma unroll
              for (int c = 0; c < 16; ++c) {
                const int col = c0 + c;
                const bool ispos = ((unsigned)(col - p0) < plen) && (col != self_col);
                const float x = __uint_as_float(v[c]) * scale;      // logit in log2 units
                const float den = ptx::ex2(x) + negi;
                acc0 += ispos ? (x - ptx::lg2(den)) : 0.f;
                acc1 += ispos ? ptx::rcp(den) : 0.f;
              }
            }
          }
        }
#ifdef MSCS_TRACE
        if (tslot > 0) { MSCS_TRACE_EV(tslot, 2, it); MSCS_TRACE_EV(tslot, 3, it); }
#endif
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&acc_empty[buf]);
        if (valid) {
          if (MODE == 0) {
            float a0, a1, b0, b1;
            ptx::unpack2(acc_a, a0, a1); ptx::unpack2(acc_b, b0, b1);
            atomicAdd(&t.neg[row], ((a0 + a1) + (b0 + b1)) + acc0);
          }
          else if (touches) { atomicAdd(&t.pos[row], acc0 * kLn2); atomicAdd(&t.ssum[row], acc1); }
        }
      }
    }
  }
  __syncwarp();
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) ptx::tmem_dealloc(tmem_base, 512);
#ifdef MSCS_TRACE
  if (MODE == MSCS_TRACE_MODE && blockIdx.x == 5 && threadIdx.x == 0) ptx::g_trace[3 * 2048 + 255 * 8 + 6] = (unsigned long long)clock64();
#endif
#ifdef MSCS_WAIT_PROFILE
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    atomicAdd(&ptx::g_wait_ns[31], ptx::globaltimer_ns() - prof_t0);
    atomicAdd(&ptx::g_wait_cnt[31], (unsigned long long)(clock64() - prof_c0));
  }
  if (threadIdx.x == 0 && blockIdx.x < 160) {
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    unsigned long long* sp = g_cta_span[MODE][blockIdx.x];
    sp[0] = prof_t0; sp[1] = ptx::globaltimer_ns(); sp[2] = (unsigned long long)(clock64() - prof_c0); sp[3] = smid;
  }
#endif
}

// per anchor row: positive key range [k_seg[y], k_seg[y+1]); per 32-row group: the union (groups are
// padded to whole 128-row tiles so the epilogue can index them by tile)
struct RangeTerm { const int* a_cls; const int* k_seg; int2* row_range; int2* grp_range; int N1; const int* n1_dev; };
struct RangeArgs { RangeTerm t[MSCS_MAX_TERMS]; double* fin_acc; };   // fin_acc: per-term loss accumulators of the finalise
__global__ void __launch_bounds__(256) k_row_ranges(const __grid_constant__ RangeArgs a) {
  pdl_trigger();
  pdl_wait();
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x < MSCS_MAX_TERMS) a.fin_acc[threadIdx.x] = 0.0;
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == MSCS_MAX_TERMS)      // the finalise kernel's ticket (simt.cu)
    *reinterpret_cast<unsigned*>(reinterpret_cast<char*>(a.fin_acc) + 1024) = 0u;
  const RangeTerm& t = a.t[blockIdx.y];
  const int r = blockIdx.x * 256 + threadIdx.x;
  const int tN1 = t.n1_dev ? *t.n1_dev : t.N1;
  if (blockIdx.x * 256 >= (tN1 + 127) / 128 * 128) return;
  int p0 = 0x7fffffff, p1 = 0;
  if (r < tN1) {
    const int y = t.a_cls[r];
    p0 = t.k_seg[y]; p1 = t.k_seg[y + 1];
    t.row_range[r] = make_int2(p0, p1);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    p0 = min(p0, __shfl_xor_sync(0xffffffffu, p0, o));
    p1 = max(p1, __shfl_xor_sync(0xffffffffu, p1, o));
  }
  if ((threadIdx.x & 31) == 0 && r < (tN1 + 127) / 128 * 128) t.grp_range[r >> 5] = make_int2(p0, p1);
}

// ---------------------------------------------------------------------------------------
// work table builder: one item per (owner, block).  MODE 0: every streamed tile; MODE 1: the
// streamed tiles whose classes overlap the classes of the block (both sides are class-sorted).
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) k_build_work(const __grid_constant__ BuildArgs a) {
  __shared__ int carry;
  __shared__ int wsum[32];
  pdl_trigger();
  pdl_wait();
  // block 1 (forward only): the table of the second sweep, built in the same launch
  const int mode = a.mode + (int)blockIdx.x;
  WorkItem* const items = blockIdx.x ? a.items1 : a.items;
  int* const prefix = blockIdx.x ? a.prefix1 : a.prefix;
  if (threadIdx.x == 0) { carry = 0; prefix[0] = 0; }
  __syncthreads();
  for (int base = 0; base < a.nitems; base += blockDim.x) {
    const int i = base + threadIdx.x;
    int len = 0;
    if (i < a.nitems) {
      int ti = 0;
      for (int q = 1; q < a.num_terms; ++q) if (i >= a.t[q].item_base) ti = q;
      const BuildTerm& t = a.t[ti];
      const int rb = t.blk_lo + i - t.item_base;
      const int tN1 = t.n1_dev ? *t.n1_dev : t.N1, tN2 = t.n2_dev ? *t.n2_dev : t.N2;
      int ct0 = 0, ct1 = (tN2 + kTileN - 1) / kTileN;
      if (rb * a.rows_per_item >= tN1) {      // block beyond the actual row count (items are sized by the upper bound)
        ct0 = ct1 = 0;
      } else if (mode == 1) {
        const int r0 = rb * a.rows_per_item, r1 = min(tN1, r0 + a.rows_per_item) - 1;
        const int p0 = t.k_seg[t.a_cls[r0]], p1 = t.k_seg[t.a_cls[r1] + 1];
        if (p1 > p0) { ct0 = p0 / kTileN; ct1 = (p1 + kTileN - 1) / kTileN; } else { ct0 = ct1 = 0; }
      }
      ct0 = max(ct0, t.ct_lo); ct1 = max(ct0, min(ct1, t.ct_hi));      // pooled mode: this rank's streamed tiles
      items[i] = WorkItem{ti, rb, ct0, ct1};
      len = ct1 > ct0 ? ct1 - ct0 + a.pad : 0;
    }
    int s = len;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int v = __shfl_up_sync(0xffffffffu, s, o); if ((threadIdx.x & 31) >= o) s += v; }
    if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
      int w = wsum[threadIdx.x], ws = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { int v = __shfl_up_sync(0xffffffffu, ws, o); if ((int)threadIdx.x >= o) ws += v; }
      wsum[threadIdx.x] = ws - w;
    }
    __syncthreads();
    const int incl = carry + wsum[threadIdx.x >> 5] + s;
    if (i < a.nitems) prefix[i + 1] = incl;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry = incl;
    __syncthreads();
  }
}

// ---- tensor map factory (driver entry point resolved at run time: no link-time libcuda) ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int make_tensor_map(CUtensorMap* out, const void* base, int rows, int c_pad) {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qr;
    MSCS_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr));
    MSCS_CHECK_ARG(p != nullptr && qr == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available");
    fn = (EncodeTiledFn)p;
  }
  cuuint64_t dims[2] = {(cuuint64_t)c_pad, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)c_pad * 2};
  cuuint32_t box[2] = {(cuuint32_t)kKBlk, 128};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = CUDA_SUCCESS;
  for (int attempt = 0; attempt < 2; ++attempt) {
    r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    // A DRIVER-API call needs a context current to the calling thread.  The backward runs on autograd's device thread,
    // and since the one-call backward (step.cu) nothing in front of it on that thread is a runtime call that would have
    // bound the primary context: bind it (cudaFree(0)) and encode again.
    if (r != CUDA_ERROR_INVALID_CONTEXT) break;
    MSCS_CUDA(cudaFree(nullptr));
  }
  MSCS_CHECK_ARG(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return 0;
}

int launch_build_work(const BuildArgs& b, cudaStream_t st) {
  MSCS_CUDA(launch_k(k_build_work, b.items1 ? 2 : 1, 1024, 0, st, b));
  MSCS_LAUNCH_CHECK();
  return 0;
}

int sm_count() {
  static int n = 0;
  if (!n) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev); }
  return n > 0 ? n : 148;
}

// Grid of the persistent tensor kernels: one CTA per SM, minus `MSCS_SPARE_SMS` (default 1, read once).  The work
// tables are cut into gridDim.x equal shares, and a CTA fills its SM (215 KB of shared memory, ~60 k registers), so a
// single foreign CTA resident anywhere -- the MT19937 generator of the next call on its side stream (sample.cu), a
// communication kernel of the training loop -- leaves 148 CTAs with 147 SMs and the kernel then lasts until a SECOND
// CTA has run on one of them.  One SM left free costs 1/148 of the tensor throughput and takes that hit away.
int persistent_ctas() {
  static const int spare = [] { const char* e = getenv("MSCS_SPARE_SMS"); const int v = e ? atoi(e) : 1; return v < 0 ? 0 : v; }();
  const int n = sm_count() - spare;
  return n > 0 ? n : 1;
}

// environment switches of the tuning experiments, read ONCE per process (no getenv on the per-step path)
struct FwdTuning { int pad; bool timeline; };
static const FwdTuning& fwd_tuning() {
  static const FwdTuning t = [] {
    FwdTuning v{0, false};
    if (const char* e = getenv("MSCS_FWD_PAD")) v.pad = atoi(e);
    v.timeline = getenv("MSCS_FWD_TIMELINE") != nullptr;
    return v;
  }();
  return t;
}

template <int KB, int MODE>
static int launch_fwd_k(const FwdArgs& args, cudaStream_t st) {
  const size_t smem = fwd_smem_bytes(KB);
  static bool attr_done = false;      // per instantiation
  if (!attr_done) {
    MSCS_CUDA(cudaFuncSetAttribute(k_sim_fwd<KB, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_done = true;
  }
  MSCS_CUDA(launch_k(k_sim_fwd<KB, MODE>, persistent_ctas(), kFwdThreads, smem, st, args));
  MSCS_LAUNCH_CHECK();
  return 0;
}

template <int KB>
static int launch_fwd(const FwdArgs& args, int mode, cudaStream_t st) {
  if (int rc = ensure_trap_buffer()) return rc;
  return mode == 1 ? launch_fwd_k<KB, 1>(args, st) : launch_fwd_k<KB, 0>(args, st);
}

}  // namespace mscs

using namespace mscs;

extern "C" size_t mscs_sim_workspace_bytes(const mscs_sim_job* job) {
  if (!job) return 0;
  size_t items = 0, ranges = 0;
  for (int t = 0; t < job->num_terms; ++t) {
    ranges += align_up(sizeof(int2) * (size_t)job->terms[t].N1, 64) +
              align_up(sizeof(int2) * (size_t)ceil_div(job->terms[t].N1, 128) * 4, 64);
    items += 2 * (size_t)ceil_div(job->terms[t].N2, kFwdKeys);                 // forward: two sweeps
    items += (size_t)ceil_div(job->terms[t].N1, 128) + ceil_div(job->terms[t].N2, 128);   // backward passes
  }
  return 2 * 4096 + ranges + items * (sizeof(WorkItem) + sizeof(int)) + 16 * 64;
}

// debug timeline (MSCS_FWD_TIMELINE=1): events after each launch of the last forward call
static cudaEvent_t g_tl[8];
static int g_tl_n = 0;
static bool g_tl_on = false;
static void tl_mark(cudaStream_t st) {
  if (!g_tl_on || g_tl_n >= 8) return;
  if (!g_tl[g_tl_n]) cudaEventCreate(&g_tl[g_tl_n]);
  cudaEventRecord(g_tl[g_tl_n++], st);
}
extern "C" int mscs_debug_fwd_timeline(float* ms_out, int max_n) {
  cudaDeviceSynchronize();
  int n = 0;
  for (int i = 1; i < g_tl_n && n < max_n; ++i, ++n) cudaEventElapsedTime(&ms_out[n], g_tl[i - 1], g_tl[i]);
  return n;
}

extern "C" int mscs_sim_forward_sweeps(const mscs_sim_job* job, void* stream_) {
  int rc = validate_job(job);
  if (rc) return rc;
  MSCS_CHECK_ARG(job->work, "work buffer is null");
  cudaStream_t st = (cudaStream_t)stream_;
  FwdArgs args{};
  g_tl_on = fwd_tuning().timeline;
  g_tl_n = 0;
  tl_mark(st);
  // one tensor map per distinct operand matrix
  const void* bases[MSCS_MAX_SCALES]; int nmaps = 0;
  auto map_of = [&](const void* base, int rows) -> int {
    for (int i = 0; i < nmaps; ++i) if (bases[i] == base) return i;
    if (nmaps == MSCS_MAX_SCALES) return -1;
    if (make_tensor_map(&args.maps[nmaps], base, (rows + 255) / 256 * 256, job->C_pad)) return -2;
    bases[nmaps] = base;
    return nmaps++;
  };
  BuildArgs b{};
  RangeArgs ra{};
  int nitems = 0, maxN1 = 0;
  char* w = (char*)job->work + 4096;      // [0,4096): finalise accumulators
  for (int t = 0; t < job->num_terms; ++t) {
    const mscs_term& m = job->terms[t];
    const int am = map_of(m.a_bf16, m.N1), km = map_of(m.k_bf16, m.N2);
    if (am == -2 || km == -2) return -1;
    MSCS_CHECK_ARG(am >= 0 && km >= 0, "too many distinct operand matrices");
    int2* rr = (int2*)w; w += align_up(sizeof(int2) * (size_t)m.N1, 64);
    int2* gr = (int2*)w; w += align_up(sizeof(int2) * (size_t)ceil_div(m.N1, 128) * 4, 64);
    ra.t[t] = RangeTerm{m.a_cls, m.k_seg, rr, gr, m.N1, m.n1_dev};
    if (m.N1 > maxN1) maxN1 = m.N1;
    args.t[t] = FwdTerm{m.a_cls, m.k_seg, rr, gr, m.neg_sum, m.pos_sum, m.s_sum, m.N1, m.N2, m.self_mask, am, km,
                        kLog2e / m.temperature, m.n1_dev, m.n2_dev};
    // blocks are on the KEY side (256 keys), the streamed 128-row tiles on the ANCHOR side
    const bool all_rows = m.row_begin == 0 && m.row_end == 0;     // 0,0 = every row; begin == end = none
    const int r_lo = all_rows ? 0 : m.row_begin, r_hi = all_rows ? m.N1 : m.row_end;
    b.t[t] = BuildTerm{m.k_cls, m.a_seg, m.N2, m.N1, nitems, 0, r_lo / 128, r_hi > r_lo ? ceil_div(r_hi, 128) : r_lo / 128,
                       m.n2_dev, m.n1_dev};      // (blocks are on the key side: rows = keys)
    nitems += ceil_div(m.N2, kFwdKeys);
  }
  ra.fin_acc = (double*)job->work;
  MSCS_CUDA(launch_k(k_row_ranges, dim3(ceil_div(maxN1 + 127, 256), job->num_terms), 256, 0, st, ra));
  MSCS_LAUNCH_CHECK();
  tl_mark(st);
  b.num_terms = job->num_terms; b.nitems = nitems; b.rows_per_item = kFwdKeys;
  b.pad = fwd_tuning().pad;      // start-up charge of a key block (128 KB load + pipeline fill), in anchor tiles
  // both work tables (sweep 0: every tile; sweep 1: class-diagonal tiles) depend only on the class arrays: one launch
  b.mode = 0;
  b.items = (WorkItem*)w;  w += align_up(sizeof(WorkItem) * (size_t)nitems, 64);
  b.prefix = (int*)w;      w += align_up(sizeof(int) * (size_t)(nitems + 1), 64);
  b.items1 = (WorkItem*)w; w += align_up(sizeof(WorkItem) * (size_t)nitems, 64);
  b.prefix1 = (int*)w;     w += align_up(sizeof(int) * (size_t)(nitems + 1), 64);
  rc = launch_build_work(b, st);
  if (rc) return rc;
  tl_mark(st);
  for (int mode = 0; mode < 2; ++mode) {
    args.work = mode ? WorkTable{b.items1, b.prefix1, nitems, b.pad} : WorkTable{b.items, b.prefix, nitems, b.pad};
    switch (job->C_pad / 64) {
      case 1: rc = launch_fwd<1>(args, mode, st); break;
      case 2: rc = launch_fwd<2>(args, mode, st); break;
      case 3: rc = launch_fwd<3>(args, mode, st); break;
      default: rc = launch_fwd<4>(args, mode, st); break;
    }
    if (rc) return rc;
    tl_mark(st);
  }
  return 0;
}

extern "C" int mscs_sim_finalize(const mscs_sim_job* job, void* stream_) {
  int rc = validate_job(job);
  if (rc) return rc;
  MSCS_CHECK_ARG(job->work, "work buffer is null");
  return launch_finalize(job, (cudaStream_t)stream_);
}

extern "C" int mscs_sim_forward(const mscs_sim_job* job, void* stream_) {
  int rc = mscs_sim_forward_sweeps(job, stream_);
  if (rc) return rc;
  rc = launch_finalize(job, (cudaStream_t)stream_);
  tl_mark((cudaStream_t)stream_);
  return rc;
}

// debug (trace build only): copy out and reset the event trace of sweep 0 of the forward kernel (CTA 5):
// [slot][tile][event] clock64 values; slot 0 = MMA warp (0 before / 1 after the acc_empty wait, 2 tile issued),
// slots 1..3 = epilogue warps 4, 11 (group 0) and 12 (group 1): 0 before / 1 after the acc_full wait, 2 math done
extern "C" int mscs_debug_trace_fwd(unsigned long long* out, int max_events) {
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

// debug (profiling build only): per-CTA spans of the last launch of sweep `mode`: 160 x {start ns, end ns, SM cycles, SM id}
extern "C" int mscs_debug_cta_spans_fwd(unsigned long long* out, int mode) {
#ifdef MSCS_WAIT_PROFILE
  MSCS_CUDA(cudaDeviceSynchronize());
  MSCS_CUDA(cudaMemcpyFromSymbol(out, g_cta_span, sizeof(unsigned long long) * 160 * 4,
                                 sizeof(unsigned long long) * 160 * 4 * (mode ? 1 : 0)));
  return 160;
#else
  (void)out; (void)mode;
  return 0;
#endif
}

// debug: read and reset the barrier wait profile of this translation unit (ns and count per tag % 32)
extern "C" int mscs_debug_wait_profile_fwd(unsigned long long* ns_out, unsigned long long* cnt_out) {
  MSCS_CUDA(cudaDeviceSynchronize());
  MSCS_CUDA(cudaMemcpyFromSymbol(ns_out, ptx::g_wait_ns, sizeof(unsigned long long) * 32));
  MSCS_CUDA(cudaMemcpyFromSymbol(cnt_out, ptx::g_wait_cnt, sizeof(unsigned long long) * 32));
  unsigned long long zero[32] = {};
  MSCS_CUDA(cudaMemcpyToSymbol(ptx::g_wait_ns, zero, sizeof(zero)));
  MSCS_CUDA(cudaMemcpyToSymbol(ptx::g_wait_cnt, zero, sizeof(zero)));
  return 0;
}
