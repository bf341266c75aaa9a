// ce.cu -- SURVEY.md section 8f item 2: the co-loss that reads the same label map as the contrastive loss.
//
// The reference's LossWrapper evaluates, next to DenseContrastiveLossV2_ms, a class-weighted
// nn.CrossEntropyLoss(ignore_index=ignore_class, weight=class_weights) over the full-resolution logits
// (losses/LossWrapper.py:22-31,81-82; TwoScaleLoss.py:62-73 applies the same loss to two logit maps).  Both losses start
// from the int64 label map.  Here ONE sweep over it (k_label_pass) produces everything either of them needs from the
// labels:
//   * compact int16 labels (-1 = outside [0, A)): what K1's down-sampling / histogram kernel and the CE kernels read
//     from then on (a quarter of the bytes, and K1 needs no int64 -> float32 -> int64 round trip any more);
//   * the full-resolution class histogram: the CE normaliser sum_valid w[y] = sum_c w[c] hist[c] is known BEFORE the
//     logits are touched, so the CE backward is a single fused pass with the final scale (no second sweep).
// The CE itself is two fused HBM-bound kernels (ATen runs log_softmax + nll_loss forward and their two backwards: about
// three times the traffic):
//   k_ce_fwd   loss_sum = sum_valid w[y] (logsumexp(x) - x_y)          reads the logits once
//   k_ce_bwd   dx_k = (g / denom) w[y] (softmax_k - [k == y]), 0 on ignored pixels   reads once (+L1), writes once
// thread = 4 consecutive pixels (float4 per class plane, 8 bytes for bf16 / fp16 logits), online max / sum over the
// classes.  Half logits are widened on load and dlogits rounded on store; the arithmetic is the fp32 kernel's.
#include "common.cuh"

namespace mscs {

constexpr int kCeMaxClasses = 1024;

// ---- one sweep over the int64 labels ------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_label_pass(const long long* __restrict__ labels, long long n_pix, int A, short* __restrict__ lab16,
             int* __restrict__ hist_out) {
  extern __shared__ int hist[];
  for (int c = threadIdx.x; c < A; c += blockDim.x) hist[c] = 0;
  __syncthreads();
  const long long stride = (long long)gridDim.x * blockDim.x * 4;
  for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < n_pix; i += stride) {
    long long v[4];
    if (i + 3 < n_pix) {
      const longlong2 a = *reinterpret_cast<const longlong2*>(labels + i);
      const longlong2 b = *reinterpret_cast<const longlong2*>(labels + i + 2);
      v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
    } else {
#pragma unroll
      for (int q = 0; q < 4; ++q) v[q] = (i + q < n_pix) ? labels[i + q] : -1;
    }
    short o[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      // the reference's contrastive path converts label -> float32 -> int64 (V2.py:205-206); class ids are far below
      // 2^24, where the round trip is the identity: the same validity test on the integer
      const bool ok = v[q] >= 0 && v[q] < A;
      o[q] = ok ? (short)v[q] : (short)-1;
      if (ok) atomicAdd(&hist[(int)v[q]], 1);
    }
    if (i + 3 < n_pix) *reinterpret_cast<short4*>(lab16 + i) = make_short4(o[0], o[1], o[2], o[3]);
    else
      for (int q = 0; q < 4 && i + q < n_pix; ++q) lab16[i + q] = o[q];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < A; c += blockDim.x)
    if (hist[c]) atomicAdd(&hist_out[c], hist[c]);
}

// denom = sum_{c < K, c != ignore} w[c] hist[c];  out = {loss_sum / denom, denom}
__global__ void k_ce_finalize(const int* __restrict__ hist, const float* __restrict__ weight, int K, int A, int ignore,
                              const double* __restrict__ loss_sum, float* __restrict__ out) {
  double d = 0.0;
  for (int c = threadIdx.x; c < K && c < A; c += 32)
    if (c != ignore) d += (double)(weight ? weight[c] : 1.f) * (double)hist[c];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
  if (threadIdx.x == 0) {
    out[0] = (float)(*loss_sum / d);      // 0/0 -> NaN when every pixel is ignored, like ATen's mean reduction
    out[1] = (float)d;
  }
}

struct CeArgs {
  const void* logits; const short* lab16; const float* weight;
  int K, plane, ignore; long long n_quads;      // quads of 4 consecutive pixels (plane % 4 == 0)
};

// online (max, sum exp) over the class planes of 4 consecutive pixels
template <typename T>
__device__ __forceinline__ void ce_stats(const T* __restrict__ base, int K, size_t plane, float (&mx)[4], float (&se)[4]) {
#pragma unroll
  for (int q = 0; q < 4; ++q) { mx[q] = -INFINITY; se[q] = 0.f; }
  for (int k = 0; k < K; ++k) {
    float xv[4];
    ld4(base + (size_t)k * plane, xv);
#pragma unroll
    for (int q = 0; q < 4; ++q) {      // one exponential per element (accurate expf: the kernels are HBM-bound)
      const float d = xv[q] - mx[q];
      if (d <= 0.f) se[q] += expf(d);
      else { se[q] = se[q] * expf(-d) + 1.f; mx[q] = xv[q]; }
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(256) k_ce_fwd(const __grid_constant__ CeArgs a, double* __restrict__ loss_sum) {
  __shared__ double red[8];
  double part = 0.0;
  const long long quad = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (quad < a.n_quads) {
    const long long pix = quad * 4;
    const long long b = pix / a.plane, p = pix - b * a.plane;
    const short4 y4 = *reinterpret_cast<const short4*>(a.lab16 + pix);
    const int y[4] = {y4.x, y4.y, y4.z, y4.w};
    bool any = false;
#pragma unroll
    for (int q = 0; q < 4; ++q) any = any || (y[q] >= 0 && y[q] < a.K && y[q] != a.ignore);
    if (any) {
      const T* base = static_cast<const T*>(a.logits) + (size_t)b * a.K * a.plane + p;
      float mx[4], se[4];
      ce_stats(base, a.K, (size_t)a.plane, mx, se);
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (y[q] >= 0 && y[q] < a.K && y[q] != a.ignore) {
          const float xy = to_f32(base[(size_t)y[q] * a.plane + q]);
          const float w = a.weight ? a.weight[y[q]] : 1.f;
          part += (double)(w * (mx[q] + logf(se[q]) - xy));
        }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < 8; ++w) s += red[w];
    if (s != 0.0) atomicAdd(loss_sum, s);
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
k_ce_bwd(const __grid_constant__ CeArgs a, const float* __restrict__ grad_out, const float* __restrict__ denom,
         T* __restrict__ dlogits) {
  const long long quad = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (quad >= a.n_quads) return;
  const long long pix = quad * 4;
  const long long b = pix / a.plane, p = pix - b * a.plane;
  const short4 y4 = *reinterpret_cast<const short4*>(a.lab16 + pix);
  const int y[4] = {y4.x, y4.y, y4.z, y4.w};
  const size_t off = (size_t)b * a.K * a.plane + p;
  const T* base = static_cast<const T*>(a.logits) + off;
  T* out = dlogits + off;
  float coef[4];
  bool any = false;
  const float g = *grad_out / *denom;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const bool ok = y[q] >= 0 && y[q] < a.K && y[q] != a.ignore;
    coef[q] = ok ? g * (a.weight ? a.weight[y[q]] : 1.f) : 0.f;
    any = any || ok;
  }
  if (!any) {      // four ignored pixels: zeros, the logits are not read
    const float z[4] = {0.f, 0.f, 0.f, 0.f};
    for (int k = 0; k < a.K; ++k) st4_cs(out + (size_t)k * a.plane, z);
    return;
  }
  float mx[4], se[4];
  ce_stats(base, a.K, (size_t)a.plane, mx, se);
  float inv[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) inv[q] = coef[q] / se[q];
  for (int k = 0; k < a.K; ++k) {
    float xv[4];
    ld4(base + (size_t)k * a.plane, xv);      // second read: L1 / L2
    float r[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) r[q] = expf(xv[q] - mx[q]) * inv[q] - (k == y[q] ? coef[q] : 0.f);
    st4_cs(out + (size_t)k * a.plane, r);
  }
}

}  // namespace mscs

using namespace mscs;

extern "C" int mscs_label_pass(const int64_t* labels, int64_t n_pixels, int num_classes, int16_t* lab16, int32_t* hist,
                               void* stream_) {
  MSCS_CHECK_ARG(labels && lab16 && hist && n_pixels >= 1, "bad arguments");
  MSCS_CHECK_ARG(num_classes >= 1 && num_classes <= 32767, "num_classes %d out of range", num_classes);
  MSCS_CHECK_ARG(((uintptr_t)labels % 16 == 0) && ((uintptr_t)lab16 % 8 == 0), "label buffers must be 16 / 8 byte aligned");
  cudaStream_t st = (cudaStream_t)stream_;
  MSCS_CUDA(cudaMemsetAsync(hist, 0, sizeof(int32_t) * num_classes, st));
  long long blocks = (n_pixels + 256 * 4 * 4 - 1) / (256 * 4 * 4);      // four quads per thread
  if (blocks > 148 * 16) blocks = 148 * 16;
  k_label_pass<<<(int)blocks, 256, sizeof(int) * num_classes, st>>>((const long long*)labels, n_pixels, num_classes, lab16,
                                                                   hist);
  MSCS_LAUNCH_CHECK();
  return 0;
}

static int ce_args(CeArgs* a, const void* logits, const int16_t* lab16, int n, int K, int plane, const float* weight,
                   int ignore_index, int dtype) {
  MSCS_CHECK_ARG(logits && lab16, "null pointer argument");
  MSCS_CHECK_ARG(dtype_bytes(dtype) > 0, "dtype %d unknown (MSCS_DTYPE_F32 / _BF16 / _F16)", dtype);
  MSCS_CHECK_ARG(n >= 1 && K >= 1 && K <= kCeMaxClasses && plane >= 4 && plane % 4 == 0,
                 "unsupported shape (n %d, K %d, plane %d: the plane must be a multiple of 4 pixels)", n, K, plane);
  const int al = 4 * dtype_bytes(dtype);      // one load / store of 4 pixels
  MSCS_CHECK_ARG((uintptr_t)logits % al == 0 && (uintptr_t)lab16 % 8 == 0, "logits / labels must be %d / 8 byte aligned",
                 al);
  a->logits = logits; a->lab16 = lab16; a->weight = weight; a->K = K; a->plane = plane; a->ignore = ignore_index;
  a->n_quads = (long long)n * plane / 4;
  return 0;
}

extern "C" int mscs_ce_forward(const void* logits, const int16_t* lab16, int n, int K, int plane, const float* weight,
                               int ignore_index, const int32_t* hist, int num_classes, double* loss_sum_scratch,
                               float* loss_and_denom, void* stream_, int dtype) {
  CeArgs a;
  if (int rc = ce_args(&a, logits, lab16, n, K, plane, weight, ignore_index, dtype)) return rc;
  MSCS_CHECK_ARG(hist && loss_sum_scratch && loss_and_denom && num_classes >= 1, "null pointer argument");
  cudaStream_t st = (cudaStream_t)stream_;
  MSCS_CUDA(cudaMemsetAsync(loss_sum_scratch, 0, sizeof(double), st));
  const unsigned grid = (unsigned)((a.n_quads + 255) / 256);
  if (dtype == MSCS_DTYPE_F32) k_ce_fwd<float><<<grid, 256, 0, st>>>(a, loss_sum_scratch);
  else if (dtype == MSCS_DTYPE_BF16) k_ce_fwd<__nv_bfloat16><<<grid, 256, 0, st>>>(a, loss_sum_scratch);
  else k_ce_fwd<__half><<<grid, 256, 0, st>>>(a, loss_sum_scratch);
  MSCS_LAUNCH_CHECK();
  k_ce_finalize<<<1, 32, 0, st>>>(hist, weight, K, num_classes, ignore_index, loss_sum_scratch, loss_and_denom);
  MSCS_LAUNCH_CHECK();
  return 0;
}

extern "C" int mscs_ce_backward(const void* logits, const int16_t* lab16, int n, int K, int plane, const float* weight,
                                int ignore_index, const float* grad_out, const float* denom, void* dlogits,
                                void* stream_, int dtype) {
  CeArgs a;
  if (int rc = ce_args(&a, logits, lab16, n, K, plane, weight, ignore_index, dtype)) return rc;
  MSCS_CHECK_ARG(grad_out && denom && dlogits && (uintptr_t)dlogits % (4 * dtype_bytes(dtype)) == 0,
                 "null / misaligned pointer argument");
  cudaStream_t st = (cudaStream_t)stream_;
  const unsigned grid = (unsigned)((a.n_quads + 255) / 256);
  if (dtype == MSCS_DTYPE_F32) k_ce_bwd<float><<<grid, 256, 0, st>>>(a, grad_out, denom, (float*)dlogits);
  else if (dtype == MSCS_DTYPE_BF16) k_ce_bwd<__nv_bfloat16><<<grid, 256, 0, st>>>(a, grad_out, denom, (__nv_bfloat16*)dlogits);
  else k_ce_bwd<__half><<<grid, 256, 0, st>>>(a, grad_out, denom, (__half*)dlogits);
  MSCS_LAUNCH_CHECK();
  return 0;
}
