// step.cu -- host orchestration of one forward / one backward in ONE C call each (single process, device-driven
// order).  Every launch below is one of the library's own entry points (sample.cu, gather.cu, sim_fwd.cu, sim_bwd.cu);
// what this file adds is their ORDER, the two-stream hand-over of the sampling chain and the optional stage events, so
// that the host mirror (the autograd.Function in _ops.py) crosses the ABI once per pass instead of eight times.
//
// forward chain (replaces, per call, DenseContrastiveLossV2_ms.forward's scale loop, _ms.py:44-82, i.e. V2.py:86-125
// sampling, V2.py:138 normalisation, V2.py:150-188 / _ms.py:113-156 loss):
//   sample stream: [wait main] [wait draws] workspace fills -> histograms / plan -> plan records copied to the host on a
//                  private stream -> selection (T, V, N read from the DEVICE plan records)
//   main stream:   optional clear of the backward's accumulators, [wait sample] gather + normalise -> similarity forward (sweeps + finalise)
//   host:          waits for the plan records only (errors, row counts for the backward); with plan_host == NULL
//                  nothing is fetched and nothing waits (CUDA graph capture: the consumers read the device records)
// backward chain (autograd backward of the same): similarity backward -> normalisation backward + dense writer.
#include "common.cuh"
#include "../../include/mscs.h"

using namespace mscs;

namespace {

// two hand-over events per (thread, device): main -> sample at the start, sample -> main after the selection
struct ChainEvents { cudaEvent_t to_sample = nullptr, to_main = nullptr; };
thread_local ChainEvents t_chain[64];

int chain_events(ChainEvents** out) {
  int dev = 0;
  MSCS_CUDA(cudaGetDevice(&dev));
  MSCS_CHECK_ARG(dev >= 0 && dev < 64, "device index %d out of range", dev);
  ChainEvents& e = t_chain[dev];
  if (!e.to_sample) {
    MSCS_CUDA(cudaEventCreateWithFlags(&e.to_sample, cudaEventDisableTiming));
    MSCS_CUDA(cudaEventCreateWithFlags(&e.to_main, cudaEventDisableTiming));
  }
  *out = &e;
  return 0;
}

inline int mark(void* ev, cudaStream_t st) {
  if (ev) MSCS_CUDA(cudaEventRecord((cudaEvent_t)ev, st));
  return 0;
}

}  // namespace

#define CHAIN(call) do { if (int rc_ = (call)) return rc_; } while (0)

extern "C" int mscs_forward_chain(const mscs_forward_chain_args* a, void* sample_stream_, void* main_stream_,
                                  mscs_scale_plan* plan_host) {
  MSCS_CHECK_ARG(a && a->cfg && a->labels && a->workspace && a->plan_dev && a->job && a->gather_items,
                 "null pointer argument");
  MSCS_CHECK_ARG(a->gather_kind >= 0 && a->gather_kind <= 1, "gather_kind %d out of range", a->gather_kind);
  cudaStream_t ss = (cudaStream_t)sample_stream_, ms = (cudaStream_t)main_stream_;
  const int S = a->cfg->num_scales;
  const bool two = ss != ms;
  ChainEvents* ev = nullptr;
  if (two) {
    CHAIN(chain_events(&ev));
    MSCS_CUDA(cudaEventRecord(ev->to_sample, ms));
    MSCS_CUDA(cudaStreamWaitEvent(ss, ev->to_sample, 0));
  }
  // cleared on the main stream, next to the (latency-bound) sampling chain instead of in front of it
  if (a->main_zero_ptr && a->main_zero_bytes) MSCS_CUDA(cudaMemsetAsync(a->main_zero_ptr, 0, a->main_zero_bytes, ms));
  if (a->wait_event) MSCS_CUDA(cudaStreamWaitEvent(ss, (cudaEvent_t)a->wait_event, 0));
  CHAIN(mark(a->stage_events[0], ss));
  if (a->n_fill > 0) CHAIN(mscs_fill_bytes(a->fill_ptrs, a->fill_values, a->fill_bytes, a->n_fill, ss));
  if (a->labels_i16)
    CHAIN(mscs_sample_plan_i16(a->cfg, (const int16_t*)a->labels, a->workspace, a->plan_dev, ss));
  else
    CHAIN(mscs_sample_plan(a->cfg, (const int64_t*)a->labels, a->workspace, a->plan_dev, ss));
  if (plan_host) CHAIN(mscs_plan_fetch_begin(a->plan_dev, S, ss));
  CHAIN(mscs_sample_select_async(a->cfg, a->plan_dev, a->v_cap, a->workspace, a->draws, a->idx_ref, a->pair_ref, a->pix,
                                 a->cls, a->seg, a->slot, ss));
  CHAIN(mark(a->stage_events[1], ss));
  if (two) {
    MSCS_CUDA(cudaEventRecord(ev->to_main, ss));
    MSCS_CUDA(cudaStreamWaitEvent(ms, ev->to_main, 0));
  }
  CHAIN(mark(a->stage_events[2], ms));
  if (a->gather_kind == 0)
    CHAIN(mscs_gather_normalize_sectors_batch((const mscs_gather_item*)a->gather_items, S, ms));
  else
    CHAIN(mscs_gather_rows_nhwc_batch((const mscs_rows_item*)a->gather_items, S, ms));
  CHAIN(mark(a->stage_events[3], ms));
  CHAIN(mscs_sim_forward(a->job, ms));
  CHAIN(mark(a->stage_events[4], ms));
  if (!plan_host) return 0;
  return mscs_plan_fetch_end(plan_host, S);      // the one host wait of the forward pass
}

extern "C" int mscs_backward_chain(const mscs_sim_job* job, const float* grad_out, float* const* dF_sets,
                                   const int32_t* dF_ld, const mscs_scatter_item* items, const int32_t* rows, int count,
                                   void* const* stage_events, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  if (stage_events) CHAIN(mark(stage_events[0], st));
  CHAIN(mscs_sim_backward(job, grad_out, dF_sets, dF_ld, st));
  if (stage_events) CHAIN(mark(stage_events[1], st));
  if (count > 0) CHAIN(mscs_scatter_dense_batch(items, rows, count, st));
  if (stage_events) CHAIN(mark(stage_events[2], st));
  return 0;
}
