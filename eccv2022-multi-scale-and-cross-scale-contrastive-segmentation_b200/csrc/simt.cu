// simt.cu -- (1) the finalise kernel (per-term loss, weighted total, backward coefficients),
// shared by every implementation; (2) plain CUDA-core fp32 versions of the similarity forward
// and backward.  The SIMT kernels are VALIDATION kernels: the tests run them next to the
// tcgen05 kernels at sizes where the CPU oracle is slow.  They take class ids per column (not
// the sorted-segment trick the tensor kernels use), so the two paths share no masking logic.
#include "sim_common.cuh"

namespace mscs {

struct FinTerm {
  const int* a_cls; const int* k_seg;
  const float* neg; const float* pos; const float* ssum;
  float* coef_s; float* coef_pn;
  int N1, self_mask; float weight;
  const int* n1_dev;      // optional device-resident row count
};
struct FinArgs { FinTerm t[MSCS_MAX_TERMS]; int num_terms; float* term_loss; float* total_loss; float* total_out; };

// loss = mean_i(-pos_i / div_i)  (V2.py:187-188, _ms.py:148-156); coefficients for K4.
// grid = (row chunks, terms): per-row work is two dependent loads deep, so it is spread over many CTAs;
// the per-term sums are reduced in fp64 (order-insensitive to far below fp32 resolution).  The LAST block to finish
// (ticket counter next to the accumulators) turns the sums into the term losses and the weighted total: one launch
// less on the critical path between the positive sweep and the backward.
__global__ void __launch_bounds__(256) k_finalize(const __grid_constant__ FinArgs a, double* acc, unsigned* ticket) {
  pdl_trigger();
  pdl_wait();
  const FinTerm& t = a.t[blockIdx.y];
  __shared__ double red[8];
  __shared__ bool last;
  double part = 0.0;
  const int base = blockIdx.x * 1024;
  const int tN1 = t.n1_dev ? *t.n1_dev : t.N1;
  if (base < tN1) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int i = base + k * 256 + threadIdx.x;
      if (i < tN1) {
        const int y = t.a_cls[i];
        const int P = t.k_seg[y + 1] - t.k_seg[y] - (t.self_mask ? 1 : 0);
        // single-scale: 0/0 -> NaN exactly like the reference; cross-scale: divisor max(P,1)
        const float div = t.self_mask ? (float)P : (float)max(P, 1);
        part += (double)(-t.pos[i] / div);
        const float invd = 1.f / (div * (float)tN1);
        t.coef_s[i] = t.ssum[i] * invd;
        t.coef_pn[i] = t.neg[i] * invd;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (base < tN1) {
      double s = 0.0;
      for (int w = 0; w < 8; ++w) s += red[w];
      atomicAdd(&acc[blockIdx.y], s);
    }
    __threadfence();
    last = atomicAdd(ticket, 1u) == gridDim.x * gridDim.y - 1;
  }
  __syncthreads();
  if (!last || threadIdx.x != 0) return;
  __threadfence();
  double total = 0.0;
  bool bad = false;
  for (int ti = 0; ti < a.num_terms; ++ti) {
    const double sum = *reinterpret_cast<volatile double*>(&acc[ti]);
    const float l = (float)(sum / (double)(a.t[ti].n1_dev ? *a.t[ti].n1_dev : a.t[ti].N1));
    a.term_loss[ti] = l;
    bad = bad || !isfinite(l);
    total += (double)a.t[ti].weight * (double)l;
  }
  a.total_loss[0] = (float)total;
  if (a.total_out) *a.total_out = (float)total;
  // device-side replacement of the logger's has_inf_or_nan(loss) host check (utils.py / LoggingManager.py:190):
  // one flag next to the scalars, fetched together with them in a single copy
  a.total_loss[1] = (bad || !isfinite((float)total)) ? 1.f : 0.f;
}

// job->work: the first 4096 bytes are reserved for these accumulators and the ticket (zeroed by k_row_ranges, the first
// kernel of the forward sweeps: no memset between the kernels of the chain)
constexpr int kFinTicketOffset = 1024;      // bytes: behind the MSCS_MAX_TERMS doubles
int launch_finalize(const mscs_sim_job* job, cudaStream_t st, bool zero_acc) {
  FinArgs a{};
  a.num_terms = job->num_terms; a.term_loss = job->term_loss; a.total_loss = job->total_loss;
  a.total_out = job->total_out;
  int maxN = 0;
  for (int t = 0; t < job->num_terms; ++t) {
    const mscs_term& m = job->terms[t];
    a.t[t] = FinTerm{m.a_cls, m.k_seg, m.neg_sum, m.pos_sum, m.s_sum, m.coef_s, m.coef_pn, m.N1, m.self_mask,
                     m.weight, m.n1_dev};
    if (m.N1 > maxN) maxN = m.N1;
  }
  double* acc = (double*)job->work;
  unsigned* ticket = (unsigned*)((char*)job->work + kFinTicketOffset);
  if (zero_acc) MSCS_CUDA(cudaMemsetAsync(acc, 0, kFinTicketOffset + sizeof(unsigned), st));
  MSCS_CUDA(launch_k(k_finalize, dim3(ceil_div(maxN, 1024), job->num_terms), 256, 0, st, a, acc, ticket));
  MSCS_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------
// SIMT forward: 64x64 logit tiles, 4x4 per thread.  MODE 0: neg sums; MODE 1: pos / S sums.
// ---------------------------------------------------------------------------------------
struct SimtFwd {
  const float* fa; const float* fk; int C;
  const int* a_cls; const int* k_cls;
  int N1, N2, self_mask; float inv_tau;
  float* neg; float* pos; float* ssum;
};

template <int MODE>
__global__ void __launch_bounds__(256) k_simt_fwd(SimtFwd t) {
  __shared__ float As[16][65], Bs[16][65];
  __shared__ float acc0[64], acc1[64];
  __shared__ int ycol[64];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int r0 = blockIdx.x * 64;
  if (tid < 64) { acc0[tid] = 0.f; acc1[tid] = 0.f; }
  int yrow[4]; float nrow[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int r = r0 + ty * 4 + i;
    yrow[i] = r < t.N1 ? t.a_cls[r] : -1;
    nrow[i] = (MODE == 1 && r < t.N1) ? t.neg[r] : 0.f;
  }
  for (int c0 = 0; c0 < t.N2; c0 += 64) {
    float acc[4][4] = {};
    __syncthreads();
    if (tid < 64) ycol[tid] = (c0 + tid < t.N2) ? t.k_cls[c0 + tid] : -2;
    for (int k0 = 0; k0 < t.C; k0 += 16) {
      for (int e = tid; e < 1024; e += 256) {
        int r = e >> 4, kk = e & 15;
        As[kk][r] = (r0 + r < t.N1 && k0 + kk < t.C) ? t.fa[(size_t)(r0 + r) * t.C + k0 + kk] : 0.f;
        Bs[kk][r] = (c0 + r < t.N2 && k0 + kk < t.C) ? t.fk[(size_t)(c0 + r) * t.C + k0 + kk] : 0.f;
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < 16; ++kk) {
        float a[4], b[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) { a[i] = As[kk][ty * 4 + i]; b[i] = Bs[kk][tx * 4 + i]; }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
      __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = r0 + ty * 4 + i;
      float p0 = 0.f, p1 = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = c0 + tx * 4 + j;
        if (r < t.N1 && c < t.N2) {
          const float l = acc[i][j] * t.inv_tau;
          const float e = expf(l);
          const bool same = ycol[tx * 4 + j] == yrow[i];
          if (MODE == 0) {
            if (!same) p0 += e;
          } else if (same && !(t.self_mask && r == c)) {
            const float den = e + nrow[i];
            p0 += l - logf(den);
            p1 += 1.f / den;
          }
        }
      }
      atomicAdd(&acc0[ty * 4 + i], p0);
      if (MODE == 1) atomicAdd(&acc1[ty * 4 + i], p1);
    }
  }
  __syncthreads();
  if (tid < 64 && r0 + tid < t.N1) {
    if (MODE == 0) t.neg[r0 + tid] = acc0[tid];
    else { t.pos[r0 + tid] = acc0[tid]; t.ssum[r0 + tid] = acc1[tid]; }
  }
}

// ---------------------------------------------------------------------------------------
// SIMT backward: per 64-row block keep X rows in smem; per 64-column tile recompute the
// logits, form W, accumulate dX += W * Y in registers (C/4 channels per thread).
// ---------------------------------------------------------------------------------------
struct SimtBwd {
  const float* fx; const float* fy; int C;
  const int* row_cls; const int* col_cls;
  const float* row_cs; const float* row_cpn; const float* row_neg;
  const float* col_cs; const float* col_cpn; const float* col_neg;
  int n_rows, n_cols, self_mask; float inv_tau, out_scale;
  const float* grad_out; float* dF; int ld;
};

__global__ void __launch_bounds__(256) k_simt_bwd(SimtBwd t) {
  extern __shared__ float sm[];
  const int C = t.C, ldc = C + 1;
  float* Xs = sm;                     // [64][C+1]
  float* Ys = Xs + 64 * ldc;          // [64][C+1]
  float* Ws = Ys + 64 * ldc;          // [64][65]
  __shared__ float ccs[64], ccpn[64], cneg[64];
  __shared__ int ycol[64];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int r0 = blockIdx.x * 64;
  for (int e = tid; e < 64 * C; e += 256) {
    int r = e / C, k = e - r * C;
    Xs[r * ldc + k] = (r0 + r < t.n_rows) ? t.fx[(size_t)(r0 + r) * C + k] : 0.f;
  }
  int yrow[4]; float rcs[4], rcpn[4], rneg[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int r = r0 + ty * 4 + i; bool ok = r < t.n_rows;
    yrow[i] = ok ? t.row_cls[r] : -1;
    rcs[i] = (ok && t.row_cs) ? t.row_cs[r] : 0.f;
    rcpn[i] = (ok && t.row_cpn) ? t.row_cpn[r] : 0.f;
    rneg[i] = (ok && t.row_neg) ? t.row_neg[r] : 1.f;
  }
  const int rr = tid >> 2, q = tid & 3;            // accumulation role: row rr, channels cc*4+q
  float acc[64];
#pragma unroll
  for (int i = 0; i < 64; ++i) acc[i] = 0.f;
  for (int c0 = 0; c0 < t.n_cols; c0 += 64) {
    __syncthreads();
    for (int e = tid; e < 64 * C; e += 256) {
      int r = e / C, k = e - r * C;
      Ys[r * ldc + k] = (c0 + r < t.n_cols) ? t.fy[(size_t)(c0 + r) * C + k] : 0.f;
    }
    if (tid < 64) {
      int c = c0 + tid; bool ok = c < t.n_cols;
      ycol[tid] = ok ? t.col_cls[c] : -2;
      ccs[tid] = (ok && t.col_cs) ? t.col_cs[c] : 0.f;
      ccpn[tid] = (ok && t.col_cpn) ? t.col_cpn[c] : 0.f;
      cneg[tid] = (ok && t.col_neg) ? t.col_neg[c] : 1.f;
    }
    __syncthreads();
    float s[4][4] = {};
    for (int k = 0; k < C; ++k) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = Xs[(ty * 4 + i) * ldc + k]; b[i] = Ys[(tx * 4 + i) * ldc + k]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) s[i][j] = fmaf(a[i], b[j], s[i][j]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int r = r0 + ty * 4 + i, c = c0 + tx * 4 + j, cj = tx * 4 + j;
        float w = 0.f;
        if (r < t.n_rows && c < t.n_cols) {
          const float e = expf(s[i][j] * t.inv_tau);
          if (ycol[cj] != yrow[i]) w = e * (rcs[i] + ccs[cj]);
          else if (!(t.self_mask && r == c)) w = -(rcpn[i] / (e + rneg[i]) + ccpn[cj] / (e + cneg[cj]));
        }
        Ws[(ty * 4 + i) * 65 + cj] = w;
      }
    __syncthreads();
    for (int j = 0; j < 64; ++j) {
      const float w = Ws[rr * 65 + j];
#pragma unroll
      for (int cc = 0; cc < 64; ++cc) {
        int ch = cc * 4 + q;
        if (ch < C) acc[cc] = fmaf(w, Ys[j * ldc + ch], acc[cc]);
      }
    }
  }
  const float sc = t.out_scale * (*t.grad_out);
  if (r0 + rr < t.n_rows)
#pragma unroll
    for (int cc = 0; cc < 64; ++cc) {
      int ch = cc * 4 + q;
      if (ch < C) atomicAdd(&t.dF[(size_t)(r0 + rr) * t.ld + ch], acc[cc] * sc);
    }
}

}  // namespace mscs

using namespace mscs;

extern "C" int mscs_debug_sim_forward_simt(const mscs_sim_job* job, const float* const* f32_sets, void* stream_) {
  int rc = validate_job(job);
  if (rc) return rc;
  MSCS_CHECK_ARG(f32_sets && job->work, "f32_sets / work is null");
  cudaStream_t st = (cudaStream_t)stream_;
  for (int mode = 0; mode < 2; ++mode)
    for (int ti = 0; ti < job->num_terms; ++ti) {
      const mscs_term& m = job->terms[ti];
      SimtFwd t{f32_sets[m.a_set], f32_sets[m.k_set], job->C_pad, m.a_cls, m.k_cls, m.N1, m.N2, m.self_mask,
                1.f / m.temperature, m.neg_sum, m.pos_sum, m.s_sum};
      MSCS_CHECK_ARG(t.fa && t.fk, "term %d: missing fp32 set", ti);
      if (mode == 0) k_simt_fwd<0><<<ceil_div(m.N1, 64), 256, 0, st>>>(t);
      else k_simt_fwd<1><<<ceil_div(m.N1, 64), 256, 0, st>>>(t);
      MSCS_LAUNCH_CHECK();
    }
  return launch_finalize(job, st, true);
}

extern "C" int mscs_debug_sim_backward_simt(const mscs_sim_job* job, const float* const* f32_sets,
                                            const float* grad_out, float* const* dF_sets, const int32_t* dF_ld,
                                            void* stream_) {
  int rc = validate_job(job);
  if (rc) return rc;
  MSCS_CHECK_ARG(f32_sets && grad_out && dF_sets && dF_ld, "null pointer argument");
  for (int t = 0; t < job->num_terms; ++t)
    MSCS_CHECK_ARG(!job->terms[t].n1_dev && !job->terms[t].n2_dev,
                   "term %d: the validation backward needs the actual row counts (n1_dev / n2_dev must be NULL)", t);
  cudaStream_t st = (cudaStream_t)stream_;
  BwdPass passes[MSCS_MAX_PASSES];
  const int np = build_passes(job, passes);
  const int C = job->C_pad;
  const size_t smem = sizeof(float) * (2 * 64 * (size_t)(C + 1) + 64 * 65);
  MSCS_CUDA(cudaFuncSetAttribute(k_simt_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  for (int i = 0; i < np; ++i) {
    const BwdPass& p = passes[i];
    SimtBwd t{f32_sets[p.row_set], f32_sets[p.col_set], C, p.row_cls, p.col_cls, p.row_cs, p.row_cpn, p.row_neg,
              p.col_cs, p.col_cpn, p.col_neg, p.n_rows, p.n_cols, p.self_mask, p.scale_log2 / kLog2e,
              p.out_scale, grad_out, dF_sets[p.row_set], dF_ld[p.row_set]};
    MSCS_CHECK_ARG(t.fx && t.fy && t.dF, "pass %d: missing buffer", i);
    k_simt_bwd<<<ceil_div(p.n_rows, 64), 256, smem, st>>>(t);
    MSCS_LAUNCH_CHECK();
  }
  return 0;
}
