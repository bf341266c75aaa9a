// common.cuh -- error plumbing and small device helpers shared by every translation unit.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/mscs.h"

namespace mscs {

// thread-local last-error string (the only mutable state in the library)
void set_error(const char* fmt, ...);
const char* get_error();

#define MSCS_CHECK_ARG(cond, ...)                                   \
  do {                                                              \
    if (!(cond)) { ::mscs::set_error(__VA_ARGS__); return -1; }     \
  } while (0)

#define MSCS_CUDA(expr)                                                                   \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      ::mscs::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                        __LINE__);                                                        \
      return (int)_e;                                                                     \
    }                                                                                     \
  } while (0)

#define MSCS_LAUNCH_CHECK()                                                               \
  do {                                                                                    \
    cudaError_t _e = cudaGetLastError();                                                  \
    if (_e != cudaSuccess) {                                                              \
      ::mscs::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e),       \
                        __FILE__, __LINE__);                                              \
      return (int)_e;                                                                     \
    }                                                                                     \
  } while (0)

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// ---- programmatic dependent launch (PDL) ------------------------------------------------------
// A step is a chain of ~19 launches, most of them a few microseconds long: with plain stream order every boundary
// costs the launch latency plus the drain of the previous grid.  Kernels launched through launch_k() carry the
// programmatic-stream-serialization attribute (unless MSCS_PDL=0): the next grid is scheduled as soon as every CTA of
// the previous one has executed pdl_trigger() (first statement of every kernel) and SM resources allow, runs its
// prologue, and blocks in pdl_wait() until the previous grid has COMPLETED and its writes are visible.  Every thread of
// every kernel executes pdl_wait() before its first global-memory access, so a grid completes only after all of its
// predecessors did (ordering stays transitive).  Launched without the attribute both instructions are no-ops.
bool pdl_enabled();        // api.cu: MSCS_PDL environment switch, read once

__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <typename... P, typename... A>
static inline cudaError_t launch_k(void (*kernel)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, A&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at{};
  at.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at.val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = &at;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<P>(args)...);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- element types of feature maps, logits and their gradients (MSCS_DTYPE_*) ---------------------------------
// Loads widen exactly to fp32, stores round to nearest even (what Tensor.to does); every kernel computes in fp32, so a
// half input gives the same fp32 values as the fp32 kernel run on its widened copy.
__device__ __forceinline__ float to_f32(float x) { return x; }
__device__ __forceinline__ float to_f32(__nv_bfloat16 x) { return __bfloat162float(x); }
__device__ __forceinline__ float to_f32(__half x) { return __half2float(x); }
template <typename T> __device__ __forceinline__ T from_f32(float x);
template <> __device__ __forceinline__ float from_f32<float>(float x) { return x; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float x) { return __float2bfloat16_rn(x); }
template <> __device__ __forceinline__ __half from_f32<__half>(float x) { return __float2half_rn(x); }

// two fp32 values -> one 32-bit word of two rounded half values (low half = a)
__device__ __forceinline__ uint32_t pack2(__nv_bfloat16*, float a, float b) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return reinterpret_cast<const uint32_t&>(h);
}
__device__ __forceinline__ uint32_t pack2(__half*, float a, float b) {
  const __half2 h = __floats2half2_rn(a, b);
  return reinterpret_cast<const uint32_t&>(h);
}

// 16 bytes of consecutive elements (4 fp32 or 8 half), streaming store
__device__ __forceinline__ void st16_cs(float* p, const float (&v)[4]) {
  __stcs(reinterpret_cast<float4*>(p), make_float4(v[0], v[1], v[2], v[3]));
}
template <typename T>
__device__ __forceinline__ void st16_cs(T* p, const float (&v)[8]) {
  const uint4 u = make_uint4(pack2(p, v[0], v[1]), pack2(p, v[2], v[3]), pack2(p, v[4], v[5]), pack2(p, v[6], v[7]));
  __stcs(reinterpret_cast<uint4*>(p), u);
}

// 4 consecutive elements (16 bytes fp32, 8 bytes half) -> fp32
__device__ __forceinline__ void ld4(const float* p, float (&v)[4]) {
  const float4 x = *reinterpret_cast<const float4*>(p);
  v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w;
}
template <typename T>
__device__ __forceinline__ void ld4(const T* p, float (&v)[4]) {
  const uint2 u = *reinterpret_cast<const uint2*>(p);
  const T* h = reinterpret_cast<const T*>(&u);
#pragma unroll
  for (int q = 0; q < 4; ++q) v[q] = to_f32(h[q]);
}
// 4 consecutive fp32 values -> 4 elements, streaming store (16 bytes fp32, 8 bytes half)
__device__ __forceinline__ void st4_cs(float* p, const float (&v)[4]) { st16_cs(p, v); }
template <typename T>
__device__ __forceinline__ void st4_cs(T* p, const float (&v)[4]) {
  __stcs(reinterpret_cast<uint2*>(p), make_uint2(pack2(p, v[0], v[1]), pack2(p, v[2], v[3])));
}

// host side: element size of an MSCS_DTYPE_* code, 0 for an unknown code
static inline int dtype_bytes(int dtype) {
  return dtype == MSCS_DTYPE_F32 ? 4 : (dtype == MSCS_DTYPE_BF16 || dtype == MSCS_DTYPE_F16) ? 2 : 0;
}

}  // namespace mscs
