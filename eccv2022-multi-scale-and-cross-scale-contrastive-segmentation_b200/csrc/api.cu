// api.cu -- library-level entry points: version, error string, device probe.
#include "common.cuh"
#include <string.h>
#include <stdlib.h>

#ifndef MSCS_PDL_DEFAULT
#define MSCS_PDL_DEFAULT 1
#endif

namespace mscs {
static thread_local char g_err[1024] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
const char* get_error() { return g_err; }

// programmatic dependent launch between the kernels of a step (common.cuh); MSCS_PDL=0 / 1 overrides the default
bool pdl_enabled() {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("MSCS_PDL");
    on = e ? (atoi(e) != 0) : MSCS_PDL_DEFAULT;
  }
  return on != 0;
}
}  // namespace mscs

static unsigned long long* g_trap_host = nullptr;
static unsigned long long* g_trap_dev = nullptr;

// host-mapped deadlock-report buffer shared by the tensor kernels (allocated on first use)
namespace mscs {
int trap_buffer_device_ptr(unsigned long long** out) {
  if (!g_trap_host) {
    unsigned long long* h = nullptr;
    MSCS_CUDA(cudaHostAlloc((void**)&h, 64 * sizeof(unsigned long long), cudaHostAllocMapped));
    memset(h, 0, 64 * sizeof(unsigned long long));
    MSCS_CUDA(cudaHostGetDevicePointer((void**)&g_trap_dev, h, 0));
    g_trap_host = h;
  }
  *out = g_trap_dev;
  return 0;
}
}  // namespace mscs

extern "C" int mscs_debug_trap_info(char* out, int len) {
  if (!out || len <= 0) return -1;
  out[0] = 0;
  if (!g_trap_host || g_trap_host[0] == 0) return 0;
  int n = (int)(g_trap_host[0] < 63 ? g_trap_host[0] : 63), off = 0;
  for (int i = 0; i < n && off < len - 64; ++i) {
    const unsigned long long r = g_trap_host[1 + i];
    off += snprintf(out + off, len - off, "[block %llu thread %llu tag %llu parity %llu] ", r >> 40, (r >> 24) & 0xffff,
                    (r >> 8) & 0xffff, r & 1);
  }
  return n;
}

extern "C" const char* mscs_version(void) { return "mscs 0.7.0 (sm_100a, tcgen05/TMA; items carry dtype; device row counts; batched raw rows; pooled half / channels-last I/O; pooled projector tail)"; }
extern "C" const char* mscs_last_error(void) { return mscs::get_error(); }
extern "C" int mscs_device_ok(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) { cudaGetLastError(); return 0; }
  int dev = 0, major = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  return major == 10;
}

// Small device -> host read on `stream` (a private copy stream), ordered after `wait_event` (may be NULL), then
// synchronised: used to read 2.5 KB of generator state back without touching the compute stream.
extern "C" int mscs_read_to_host(void* dst_host, const void* src_dev, size_t bytes, void* wait_event, void* stream_) {
  MSCS_CHECK_ARG(dst_host && src_dev && bytes > 0, "bad arguments");
  cudaStream_t st = (cudaStream_t)stream_;
  if (wait_event) MSCS_CUDA(cudaStreamWaitEvent(st, (cudaEvent_t)wait_event, 0));
  MSCS_CUDA(cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, st));
  MSCS_CUDA(cudaStreamSynchronize(st));
  return 0;
}

// Up to four byte-fills in one call (workspace initialisation of a step: statistics = 0, slot map = -1, ...).
extern "C" int mscs_fill_bytes(void* const* ptrs, const int32_t* values, const size_t* bytes, int count, void* stream_) {
  MSCS_CHECK_ARG(ptrs && values && bytes && count >= 0 && count <= 8, "bad arguments");
  for (int i = 0; i < count; ++i)
    if (bytes[i]) MSCS_CUDA(cudaMemsetAsync(ptrs[i], values[i], bytes[i], (cudaStream_t)stream_));
  return 0;
}

