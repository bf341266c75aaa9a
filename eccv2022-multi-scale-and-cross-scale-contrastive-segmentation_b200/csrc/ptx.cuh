// ptx.cuh -- raw sm_100a PTX wrappers: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA,
// TMEM alloc/ld, commit, fences) and the UMMA shared-memory / instruction descriptors.
// Descriptor bit layouts follow the PTX ISA "tcgen05 matrix descriptors" tables.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace mscs {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// one lane of a fully active warp (elect.sync): ptxas then knows exactly one lane runs the guarded
// uniform-datapath instructions (UTCHMMA / UTMALDG) and emits no per-instruction broadcast loop
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---- mbarrier ---------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Deadlock guard: a wait that does not complete within ~2 s records (block, thread, tag, parity)
// in a host-mapped buffer and traps, so a protocol bug surfaces as a launch error with a
// diagnosis instead of hanging the GPU.  (The record is readable after the trap: it lives in
// pinned host memory, see mscs_debug_trap_info.)
static __device__ unsigned long long* g_trap_buf = nullptr;   // one copy per translation unit
// wait profile: nanoseconds spent in the slow path of mbar_wait per tag (tag % 32), summed over all threads
static __device__ unsigned long long g_wait_ns[32];
static __device__ unsigned long long g_wait_cnt[32];
// event trace (make trace, -DMSCS_TRACE): lane 0 of selected warps of ONE CTA records (event, tile, clock64)
#ifdef MSCS_TRACE
static __device__ unsigned long long g_trace[8192];       // [4 slots][256 tiles][8 events] clock64 values
#define MSCS_TRACE_EV(slot, k, tile)                                                                 \
  do {                                                                                               \
    if (blockIdx.x == 5 && (threadIdx.x & 31) == 0 && (tile) < 256u)                                 \
      mscs::ptx::g_trace[(slot) * 2048 + (tile) * 8 + (k)] = (unsigned long long)clock64();          \
  } while (0)
#else
#define MSCS_TRACE_EV(slot, k, tile) do { } while (0)
#endif
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
static __device__ __noinline__ void mbar_wait_slow(uint64_t* bar, uint32_t parity, uint32_t tag) {
  // plain retries first: reading %globaltimer costs a few hundred cycles, which showed up as wake-up latency on
  // every wait that was entered before its barrier completed (try_wait itself suspends the thread in hardware)
  for (int i = 0; i < 64; ++i)
    if (mbar_try_wait(bar, parity)) return;
  const unsigned long long t0 = globaltimer_ns();
  while (!mbar_try_wait(bar, parity)) {
    if (globaltimer_ns() - t0 > 2000000000ull) {
      if (g_trap_buf != nullptr) {
        const unsigned long long slot = atomicAdd(&g_trap_buf[0], 1ull);
        if (slot < 63)
          g_trap_buf[1 + slot] = ((unsigned long long)blockIdx.x << 40) | ((unsigned long long)threadIdx.x << 24) |
                                 ((unsigned long long)(tag & 0xffffu) << 8) | (parity & 1u);
        __threadfence_system();
      }
      __trap();
    }
  }
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, uint32_t tag = 0) {
#ifdef MSCS_WAIT_PROFILE     // profiling build (make prof): time every wait, including the first probe
  const unsigned long long t0 = globaltimer_ns();
  if (!mbar_try_wait(bar, parity)) mbar_wait_slow(bar, parity, 0);
  atomicAdd(&g_wait_ns[tag & 31], globaltimer_ns() - t0);
  atomicAdd(&g_wait_cnt[tag & 31], 1ull);
#else
  if (mbar_try_wait(bar, parity)) return;
  mbar_wait_slow(bar, parity, tag);
#endif
}

// Low-latency wait for the thread that feeds the tensor pipe: polls with the NON-blocking test_wait.  A thread
// suspended inside try_wait resumed ~250 cycles after the phase completed (measured, tools/trace_bwd.py) -- longer
// than the work the pipe has buffered, i.e. a bubble on every tile.  Falls back to the guarded wait.
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_spin_wait(uint64_t* bar, uint32_t parity, uint32_t tag) {
#ifdef MSCS_WAIT_PROFILE
  mbar_wait(bar, parity, tag);
#else
  for (int i = 0; i < 4096; ++i)
    if (mbar_test_wait(bar, parity)) return;
  mbar_wait(bar, parity, tag);
#endif
}

// ---- fences -----------------------------------------------------------------------------
__device__ __forceinline__ void fence_proxy_async_smem() {   // generic-proxy smem writes -> async proxy (UMMA/TMA)
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- TMA --------------------------------------------------------------------------------
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2D tile load global -> shared, completion on an mbarrier (bytes)
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int x, int y) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(x), "r"(y)
      : "memory");
}

// ---- TMEM -------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_out, uint32_t ncols) {   // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_out)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {      // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// 32 lanes x 32 consecutive 32-bit columns: thread t of the warp gets lane (base_lane + t)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
// 32 lanes x 16 consecutive 32-bit columns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait16(uint32_t (&v)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15])
               :
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// wait for outstanding tcgen05.ld and tie the destination registers to the wait, so the
// compiler cannot schedule a use of them above it
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&v)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]), "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]), "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
               :
               : "memory");
}

// 32 lanes x 16 consecutive 32-bit columns, registers -> TMEM
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
        "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
               "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
        "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),
        "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]),
        "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- UMMA -------------------------------------------------------------------------------
// shared-memory matrix descriptor, 128-byte swizzle.  Operand tiles are stored as [rows][64 bf16]
// (128 B per row, 8-row groups of 1024 B), exactly what a TMA box {64, rows} with SWIZZLE_128B writes.
//   K-major  use (rows = M/N index, the 128 B row runs along K): SBO = 1024 (next 8 rows), LBO unused
//   MN-major use (rows = K index, the 128 B row runs along M/N): SBO = 1024 (next 8 K rows),
//                                                                LBO = byte stride to the next 64 M/N elements
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;   // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;   // SWIZZLE_128B
  return d;
}
// instruction descriptor, kind::f16, bf16 x bf16 -> fp32
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread
__device__ __forceinline__ void umma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]: A is M=128 lanes x K, 16-bit elements packed two per 32-bit column
// (element 2c in the low half of column c) -- layout verified on hardware by tools/umma_probe.cu
__device__ __forceinline__ void umma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same MMAs with the 64-bit shared-memory descriptors passed as (lo, hi) halves.  The tensor pipe executes a
// 128 x N x 16 MMA in N/2 cycles, so for N <= 128 the ISSUE code must cost less than that per MMA: with the
// descriptor of a tile precomputed once, stepping to the next K slice / K block is ONE 32-bit add on `lo`
// (the start-address field, 16-byte units; all operand offsets here stay below its 256 KB range).
__device__ __forceinline__ void umma_ts2(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 bd;\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 bd, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], bd, %4, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_ss2(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                         uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 ad, bd;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 ad, {%1, %2};\n\t"
      "mov.b64 bd, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], ad, bd, %5, p;\n\t}"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// make an mbarrier track completion of all previously issued MMAs of this thread
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// 2^(v*scale) on the FMA / ALU pipes only (no MUFU): round-to-nearest split x = n + f with the
// 1.5*2^23 trick, degree-4 minimax polynomial of 2^f on [-0.5, 0.5] (max relative error 2.7e-6),
// n added into the exponent field.  Valid for |v*scale| < 120.  Used to take part of the exp
// load off the 16/clk/SM MUFU unit in the forward epilogue.
__device__ __forceinline__ float ex2_poly(float v, float scale) {
  const float magic = 12582912.f;
  const float t = fmaf(v, scale, magic);
  const float n = t - magic;
  const float f = fmaf(v, scale, -n);
  float p = fmaf(0.009570100344717503f, f, 0.05591785907745361f);
  p = fmaf(p, f, 0.240247443318367f);
  p = fmaf(p, f, 0.6931217908859253f);
  p = fmaf(p, f, 0.9999992847442627f);
  return __int_as_float(__float_as_int(p) + (__float_as_int(t) << 23));
}
// ---- packed fp32x2 arithmetic (sm_100: one FMA-pipe issue slot for two elements) -------------
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ uint64_t pack2u(uint32_t lo, uint32_t hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
// two exponentials 2^(v*scale) per call, polynomial path (see ex2_poly), packed arithmetic:
// 7 FMA-pipe instructions + 2 integer adds for two elements
__device__ __forceinline__ uint64_t ex2_poly2(uint64_t v, uint64_t scale2) {
  const uint64_t magic = pack2(12582912.f, 12582912.f), nmagic = pack2(-12582912.f, -12582912.f);
  const uint64_t t = fma2(v, scale2, magic);
  const uint64_t n = add2(t, nmagic);
  const uint64_t nn = n ^ 0x8000000080000000ull;          // -n (sign flips fold into the operand modifiers)
  const uint64_t f = fma2(v, scale2, nn);
  uint64_t p = fma2(pack2(0.009570100344717503f, 0.009570100344717503f), f, pack2(0.05591785907745361f, 0.05591785907745361f));
  p = fma2(p, f, pack2(0.240247443318367f, 0.240247443318367f));
  p = fma2(p, f, pack2(0.6931217908859253f, 0.6931217908859253f));
  p = fma2(p, f, pack2(0.9999992847442627f, 0.9999992847442627f));
  const uint32_t plo = (uint32_t)p, phi = (uint32_t)(p >> 32), tlo = (uint32_t)t, thi = (uint32_t)(t >> 32);
  return pack2u(plo + (tlo << 23), phi + (thi << 23));
}
__device__ __forceinline__ float lg2(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

}  // namespace ptx
}  // namespace mscs
