/*
 * mscs.h -- C ABI of libmscs.so: the B200 (sm_100a) implementation of the multi-scale and
 * cross-scale dense supervised contrastive loss.
 *
 * The reference has no FFI: the loss is plain Python/ATen, dispatched by class name from
 * losses/LossWrapper.py:33,68-71.  This header is the boundary a binding would use; the
 * Python host side (mscs_b200/losses.py, _ops.py) mirrors the reference classes on top of it
 * through ctypes.  Every entry point cites the reference code it replaces.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing blocks
 *     except mscs_plan_fetch (one small D2H + stream synchronise);
 *   - every function returns 0 on success, <0 for an invalid argument, >0 for a cudaError_t;
 *     mscs_last_error() returns a thread-local message for the last failure;
 *   - memory is owned by the caller (the host side allocates workspaces with the sizes
 *     mscs_*_bytes report); the library keeps no global mutable state.
 */
#ifndef MSCS_H_
#define MSCS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSCS_MAX_SCALES 8
#define MSCS_MAX_TERMS 16   /* single-scale terms + cross-scale terms */
#define MSCS_MAX_PASSES 32  /* backward passes: 1 per ms term, up to 2 per cs term */
#define MSCS_MAX_RANKS 8    /* pooled mode: GPUs of one box */
#define MSCS_IPC_HANDLE_BYTES 64

/* element type of a feature map / its dense gradient (the `dtype` member of the gather / rows / scatter items) and of
 * the CE logits / dlogits.  Half inputs are widened exactly to fp32 on load; all arithmetic is fp32; half outputs are
 * rounded to nearest even on store (the rounding of torch's Tensor.to). */
#define MSCS_DTYPE_F32 0
#define MSCS_DTYPE_BF16 1
#define MSCS_DTYPE_F16 2

/* library info ------------------------------------------------------------------------- */
const char* mscs_version(void);
const char* mscs_last_error(void);
/* after a launch failure: textual record of barrier waits that timed out inside the tensor kernels
 * (block, thread, wait tag); returns the number of records */
int mscs_debug_trap_info(char* out, int len);
/* debug: read + reset the time spent in barrier waits inside the forward / backward tensor kernels,
 * 32 entries indexed by wait tag % 32 (nanoseconds summed over threads, and wait counts) */
int mscs_debug_wait_profile_fwd(unsigned long long* ns_out, unsigned long long* cnt_out);
int mscs_debug_wait_profile_bwd(unsigned long long* ns_out, unsigned long long* cnt_out);
/* debug (library built with -DMSCS_TRACE only, otherwise returns 0): copy out and reset the event trace of
   the backward tensor kernel -- clock64 values of one CTA, indexed [4 slots][256 tiles][8 events]. */
int mscs_debug_trace_bwd(unsigned long long* out, int max_events);
/* the same for sweep 0 of the forward tensor kernel (slot 0 = MMA warp, slots 1..3 = three epilogue warps) */
int mscs_debug_trace_fwd(unsigned long long* out, int max_events);
/* debug (MSCS_FWD_TIMELINE set in the environment): milliseconds between the launches of the last forward call
   (row ranges, work table 0, sweep 0, work table 1, sweep 1); returns the number of intervals */
int mscs_debug_fwd_timeline(float* ms_out, int max_n);
/* profiling build (make prof) only: per-CTA spans of the last launch of forward sweep `mode`:
   160 x {start ns, end ns, SM cycles, SM id}; returns 160 (0 in the product build) */
int mscs_debug_cta_spans_fwd(unsigned long long* out, int mode);
/* 1 if a CUDA device with compute capability 10.x is present */
int mscs_device_ok(void);
/* up to 8 asynchronous byte fills in one call (per-step workspace initialisation: statistics = 0, slot maps = 0xFF) */
/* small device->host read on `stream`, ordered after `wait_event` (cudaEvent_t or NULL), synchronised before return */
int mscs_read_to_host(void* dst_host, const void* src_dev, size_t bytes, void* wait_event, void* stream);
int mscs_fill_bytes(void* const* ptrs, const int32_t* values, const size_t* bytes, int count, void* stream);

/* ---------------------------------------------------------------------------------------
 * K1 -- sampling.  Replaces get_dist_and_classes (DenseContrastiveLossV2.py:194-206),
 * sample_anchors_fast (:86-125) and _select_views_per_class (:64-84) for ALL scales of one
 * call in one go.  Bit-exact with the reference given the MT19937 state of the torch CPU
 * default generator at the time of the call.
 * ------------------------------------------------------------------------------------- */
typedef struct {
  int32_t n, H, W;               /* label map (n,H,W) int64                                */
  int32_t num_scales;
  int32_t fh[MSCS_MAX_SCALES];   /* feature map height / width per scale                   */
  int32_t fw[MSCS_MAX_SCALES];
  int32_t num_classes;           /* A = num_all_classes (V2.py:16); last column is dropped  */
  int32_t min_views;             /* min_views_per_class (V2.py:21)                         */
  int32_t max_views;             /* max_views_per_class (V2.py:27); 1 = no cap (V2.py:65)  */
  int32_t max_total;             /* max_features_total (V2.py:28)                          */
  /* pooled cross-batch mode (one process per GPU, each with n local images): total number of
   * images over all ranks and the global index of this rank's first image.  0/0 = single process. */
  int32_t n_global;
  int32_t image_base;
} mscs_sample_cfg;

/* per-scale result header, written by the plan kernel, fetched by mscs_plan_fetch */
typedef struct {
  int32_t T;          /* kept (image,class) pairs                       (V2.py:111) */
  int32_t V;          /* views per pair                                  (V2.py:64-84) */
  int32_t N;          /* T*V anchors                                                 */
  int32_t min_count;  /* min pixel count over kept pairs                 (V2.py:110) */
  int32_t log_flag;   /* log_this_step as the reference sets it          (V2.py:75,83) */
  int32_t dl_h, dl_w; /* down-sampled label size (H//s, W//s), s = W//fw (V2.py:46,205) */
  int32_t error;      /* 0 ok, 1 = no pair kept, 2 = a kept pair has a single pixel, 3 = V > 16384 (N is 0 then) */
  int64_t draw_base;  /* offset of this scale's first draw in the MT19937 stream     */
  int64_t draws;      /* sum over kept pairs of (count-1)                            */
} mscs_scale_plan;

/* bytes of device workspace K1 needs for this configuration (labels, histograms, plan) */
size_t mscs_sample_workspace_bytes(const mscs_sample_cfg* cfg);
/* upper bound of MT19937 draws one call can consume (sizes the stream buffer, uint32 each) */
size_t mscs_sample_max_draws(const mscs_sample_cfg* cfg);

/* Phase 1 (async): down-sample, histogram, plan.  `plan_dev` receives num_scales
 * mscs_scale_plan records. */
int mscs_sample_plan(const mscs_sample_cfg* cfg, const int64_t* labels, void* workspace,
                     mscs_scale_plan* plan_dev, void* stream);
/* The two halves of mscs_sample_plan, for the pooled mode: (1) local down-sampling + histograms;
 * the per-(image,class) counts of scale s sit at byte offset mscs_sample_counts_offset(cfg, s) of the
 * workspace as int32 [n][A], to be all-gathered by the caller; (2) the plan from the all-gathered
 * counts int32 [n_global][A] per scale (NULL = use the local counts, single process). */
size_t mscs_sample_counts_offset(const mscs_sample_cfg* cfg, int scale);
int mscs_sample_hist(const mscs_sample_cfg* cfg, const int64_t* labels, void* workspace, void* stream);
int mscs_sample_plan_from_counts(const mscs_sample_cfg* cfg, const int32_t* const* counts_global, void* workspace,
                                 mscs_scale_plan* plan_dev, void* stream);
/* D2H of the plan records + stream synchronise (the one host sync of the forward pass;
 * the reference has ~1000, SURVEY.md §3.2). */
int mscs_plan_fetch(const mscs_scale_plan* plan_dev, mscs_scale_plan* plan_host, int num_scales,
                    void* stream);
/* The same fetch split in two, so that work enqueued in between overlaps the host wait: begin = async copy into a
 * pinned staging buffer, ordered after what `stream` holds at the call but executed on a private stream (work enqueued
 * on `stream` afterwards does not queue behind the copy); end = wait for that copy only, then hand the records out.
 * (One outstanding fetch per host thread.) */
int mscs_plan_fetch_begin(const mscs_scale_plan* plan_dev, int num_scales, void* stream);
int mscs_plan_fetch_end(mscs_scale_plan* plan_host, int num_scales);
/* MT19937 stream (async): `n_words` consecutive UNTEMPERED state words (the consumer applies the
 * tempering) of the generator whose state is
 * (mt_state_host[624], mt_pos in 0..624) -- the torch CPU default generator, which the reference
 * consumes through torch.randperm (V2.py:121).  draws_dev must hold n_words + 1024 words.  It only
 * depends on the generator state, so the host side produces it ahead of time on a side stream. */
int mscs_mt19937_stream(const uint32_t* mt_state_host, int mt_pos, uint64_t n_words, uint32_t* draws_dev,
                        void* stream);
/* Opt-in counter-based stream (not a reference behaviour; SURVEY.md 8f item 4): `n_words` words of Philox4x32-10,
 * word j = philox(counter = (j >> 2, 0, call lo, call hi), key = (seed lo, seed hi))[j & 3], stored in the same
 * buffer convention as mscs_mt19937_stream (the selection kernel tempers what it reads, so the words are stored through
 * the inverse tempering).  draws_dev: 16-byte aligned, n_words rounded up to a multiple of 4 words. */
int mscs_philox_stream(uint64_t seed, uint64_t call, uint64_t n_words, uint32_t* draws_dev, void* stream);
/* The same with the call index in DEVICE memory (a CUDA graph replays it unchanged): the words of
 * mscs_philox_stream(seed, *call_dev, ...), then *call_dev += 1 in a one-thread launch behind the generator on `stream`.
 * call_dev: 8-byte aligned. */
int mscs_philox_stream_dev(uint64_t seed, uint64_t* call_dev, uint64_t n_words, uint32_t* draws_dev, void* stream);
/* Phase 2 (async): per-pair Fisher-Yates prefix + rank->pixel selection from a precomputed stream.
 *   draws_dev : MT19937 stream starting at the generator position of this call;
 * outputs per scale s (arrays of N_s entries, N_s from the fetched plan):
 *   idx_ref[s]  : flat pixel index y*w+x in REFERENCE order k*V+v            (V2.py:122)
 *   pair_ref[s] : (T,2) int32 (image, class) in reference order              (V2.py:106-107)
 *   pix[s]      : image*fh*fw + y*dl_w+x (global pixel id in FEATURE planes, V2.py:97,123), rows sorted by class
 *   cls[s]      : class id of each sorted row
 *   seg[s]      : A+1 int32, seg[c] = first sorted row of class c, seg[A] = N
 *   slot[s]     : optional (array or entries may be NULL): int32 n*fh*fw pixel -> sorted row map,
 *                 PRE-FILLED with -1 by the caller; the sampled pixels receive their row
 */
int mscs_sample_select(const mscs_sample_cfg* cfg, const mscs_scale_plan* plan_host, void* workspace,
                       const uint32_t* draws_dev, int32_t* const* idx_ref, int32_t* const* pair_ref,
                       int32_t* const* pix, int32_t* const* cls, int32_t* const* seg, int32_t* const* slot,
                       void* stream);
/* Selection driven by the DEVICE plan records (T, V, draw offsets read in the kernel): can be enqueued before the
 * host has fetched the plan.  `v_cap`: upper bound of views per pair for this configuration (sizes shared memory). */
int mscs_sample_select_async(const mscs_sample_cfg* cfg, const mscs_scale_plan* plan_dev, int v_cap, void* workspace,
                             const uint32_t* draws_dev, int32_t* const* idx_ref, int32_t* const* pair_ref,
                             int32_t* const* pix, int32_t* const* cls, int32_t* const* seg, int32_t* const* slot,
                             void* stream);
/* host helper: advance an MT19937 state by k draws exactly as at::mt19937 does */
int mscs_mt19937_advance_host(uint32_t* mt_state_host, int* mt_pos, uint64_t k);

/* ---------------------------------------------------------------------------------------
 * K2 -- gather + L2 normalise.  Replaces the strided gather features[b,:,idx] (V2.py:123)
 * and F.normalize(p=2, dim=1) (V2.py:138, _ms.py:95,104).
 *   feat : NCHW (n,C,fh,fw) contiguous, fp32 (the batched form also bf16 / fp16, see `dtype`);  pix/N from K1
 *   anc_bf16 : (N_pad, C_pad) bf16 row-major, C_pad = C rounded up to 64, N_pad = N rounded
 *              up to 256; padding is written as zeros   (operand of the similarity kernels)
 *   anc_f32  : (N, C) fp32 unit rows (used by the normalisation backward)
 *   inv_norm : (N) 1/max(||x||, 1e-12)
 * ------------------------------------------------------------------------------------- */
int mscs_gather_normalize(const float* feat, int n, int C, int plane, const int32_t* pix, int N,
                          void* anc_bf16, float* anc_f32, float* inv_norm, void* stream);
/* same result, driven by the slot map (pixel -> row) in ADDRESS order, which keeps the strided sector
 * reads inside open DRAM pages; needs plane % 8 == 0 */
int mscs_gather_normalize_sectors(const float* feat, int n, int C, int plane, const int32_t* slot, int N,
                                  void* anc_bf16, float* anc_f32, float* inv_norm, void* stream);
/* every scale of a call in ONE launch, device-driven: the row count is read from device memory (`n_rows_dev`, e.g.
 * &plan_dev[s].N) and the padding rows are zeroed inside the call.  `dtype` (MSCS_DTYPE_*, last member: a
 * zero-initialised item is fp32) is the element type of `feat`; scales of different dtypes may be mixed (one launch
 * per dtype present).  The outputs are the same for a half map and for its exact fp32 widening. */
typedef struct {
  const void* feat; int32_t n, C, plane; const int32_t* slot; const int32_t* n_rows_dev;
  void* anc_bf16; float* anc_f32; float* inv_norm;
  int32_t dtype;
} mscs_gather_item;
int mscs_gather_normalize_sectors_batch(const mscs_gather_item* items, int count, void* stream);

/* ---------------------------------------------------------------------------------------
 * K3 / K4 -- fused similarity + loss forward and backward for every term of one call.
 * Replaces contrastive_loss/get_masks2/get_loss (V2.py:127-192), the cross-scale
 * contrastive_loss/InfoNce_loss (_ms.py:84-161), the weighted combination (_ms.py:51-80)
 * and the autograd backward of all of it.  The N x N logits are never materialised.
 * ------------------------------------------------------------------------------------- */
typedef struct {
  /* anchors (rows) and keys (columns); for a single-scale term they are the same set */
  const void* a_bf16; const void* k_bf16;   /* (N_pad, C_pad) bf16                     */
  const int32_t* a_cls; const int32_t* k_seg; /* row classes; key class segments (A+1)  */
  const int32_t* k_cls; const int32_t* a_seg; /* used by the key-side backward pass      */
  int32_t N1, N2;
  int32_t self_mask;      /* 1: single-scale term (V2.py:164-170), 0: cross-scale (_ms.py:128) */
  int32_t need_dk;        /* 0 when the key side is detached (_ms.py:66-67) or self_mask */
  float temperature;
  float weight;           /* weights[s] / w_high_low / w_high_mid  (_ms.py:54,72,79)     */
  int32_t a_set, k_set;   /* which anchor set (scale) rows/cols belong to: grads accumulate per set */
  /* pooled mode: the anchor rows [row_begin, row_end) this rank computes statistics and gradients for,
   * and the key rows [krow_begin, krow_end) whose key-side gradient it computes (cross-scale terms).
   * Multiples of 128 (the ends may equal N1 / N2).  0,0 = all rows. */
  int32_t row_begin, row_end, krow_begin, krow_end;
  /* per-anchor statistics, N1 floats each, zero-initialised by the caller */
  float* neg_sum;   /* sum_k neg exp(l_ik)                          (V2.py:183-184) */
  float* pos_sum;   /* sum_j pos [l_ij - log(e^l_ij + neg_i)]       (V2.py:186-187) */
  float* s_sum;     /* sum_j pos 1/(e^l_ij + neg_i)     (backward, SURVEY.md App. A) */
  float* coef_s;    /* out: S_i/(div_i N1)  */
  float* coef_pn;   /* out: neg_i/(div_i N1) */
  /* Optional: the row counts live in DEVICE memory (e.g. &plan_dev[s].N).  N1 / N2 above are then UPPER BOUNDS (they
   * size grids, work tables and tensor maps) and the kernels read the actual counts, so the forward and the backward
   * can be enqueued before the host has seen the sampling plan (or without it ever doing so: CUDA graphs).  NULL = N1 /
   * N2 are the actual counts.  The backward takes them for every term or for none; a count of 0 gives an empty pass.
   * Rows [count, count rounded up to 256) of the operand matrix must be ZERO, as the gathers write them: the kernels
   * load whole 128-row tiles and 256-key blocks, and the backward keeps the row coefficient of a column at or beyond
   * the count (W = e * cS_i != 0), so those columns add nothing only because their rows are zero.  Rows at or above
   * the count rounded up to 256 are never read, and class ids at or above the count are never read.  Statistics and
   * coefficients of rows at or above the count are not written, gradient rows there are not touched. */
  const int32_t* n1_dev; const int32_t* n2_dev;
} mscs_term;

typedef struct {
  int32_t num_terms;
  int32_t C_pad;
  int32_t num_classes;
  mscs_term terms[MSCS_MAX_TERMS];
  float* term_loss;   /* out: num_terms floats, unweighted per-term losses (ms_losses/cs_losses) */
  float* total_loss;  /* out: 2 floats: [0] = sum_t weight_t * term_loss_t; [1] = 1.0 if any term or the
                         total is inf/NaN else 0.0 (device-side has_inf_or_nan, LoggingManager.py:190) */
  void* work;         /* scratch, mscs_sim_workspace_bytes() */
  float* total_out;   /* optional out (NULL = unused): a second copy of total_loss[0] in a buffer of its own -- the
                         0-d tensor handed to the caller, which LossWrapper.py:90 multiplies IN PLACE (`loss *= w`):
                         it must not alias the logged scalars above (nor be a view of them for autograd) */
} mscs_sim_job;

size_t mscs_sim_workspace_bytes(const mscs_sim_job* job);
/* forward: negative sweep, positive sweep, finalise (loss + backward coefficients) */
int mscs_sim_forward(const mscs_sim_job* job, void* stream);
/* the same in two halves for the pooled mode: the sweeps over this rank's anchor rows, then (after the
 * caller has all-reduced the row statistics) the finalisation over all rows */
int mscs_sim_forward_sweeps(const mscs_sim_job* job, void* stream);
int mscs_sim_finalize(const mscs_sim_job* job, void* stream);
/* backward: dF[set] (N_set, C) fp32 += d total_loss / d unit rows * (*grad_out), for every
 * set; the caller zero-initialises dF.  grad_out is a device scalar (upstream gradient).  With device-resident row
 * counts (mscs_term.n1_dev / n2_dev) only the rows below the counts are written. */
int mscs_sim_backward(const mscs_sim_job* job, const float* grad_out, float* const* dF_sets,
                      const int32_t* dF_ld, void* stream);
/* the same restricted to the passes whose row set s has bit s of `set_mask` set (pooled mode: one launch per
 * set, so that the exchange of a set's gradient rows overlaps the tensor work of the next set) */
int mscs_sim_backward_sets(const mscs_sim_job* job, const float* grad_out, float* const* dF_sets,
                           const int32_t* dF_ld, uint32_t set_mask, void* stream);
/* plain CUDA-core fp32 versions of the two calls above: validation kernels for the tests,
 * never used by the product path */
int mscs_debug_sim_forward_simt(const mscs_sim_job* job, const float* const* f32_sets, void* stream);
int mscs_debug_sim_backward_simt(const mscs_sim_job* job, const float* const* f32_sets,
                                 const float* grad_out, float* const* dF_sets, const int32_t* dF_ld,
                                 void* stream);

/* ---------------------------------------------------------------------------------------
 * Scatter -- normalisation backward + dense gradient.  Replaces the autograd backward of
 * F.normalize and of the CopySlices/index gather (V2.py:123,138): writes the full dense
 * (n,C,fh,fw) gradient: zeros everywhere except the sampled pixels.
 * ------------------------------------------------------------------------------------- */
int mscs_scatter_grad(const float* dF, int ldF, const float* anc_f32, const float* inv_norm,
                      const int32_t* pix, int N, int n, int C, int plane, float* dfeat,
                      int zero_fill, void* stream);

/* Scatter when the caller has ALREADY zero-filled dfeat (the host side does that
 * on a side stream while the tensor kernels run) and plane % 8 == 0:
 *   mscs_slot_map              slot[image*plane + pixel] = sorted anchor row sampled there, else -1
 *   mscs_scatter_sectors_batch rewrites, with full 32-byte sector stores, only the sectors of dfeat that
 *                              hold a sampled pixel (same maths as mscs_scatter_grad). */
int mscs_slot_map(const int32_t* pix, int N, int n_pixels, int32_t* slot, void* stream);
/* every scale of a call in ONE launch.  `dtype` (MSCS_DTYPE_*): element type of `dfeat`; the gradient rows dF stay
 * fp32.  mscs_scatter_sectors_batch takes fp32 items only.  `n_rows_dev` (last member, mscs_scatter_dense_batch only):
 * NULL = `rows[s]` is the row count; else the count is read from device memory (e.g. &plan_dev[s].N) and `rows[s]` is
 * its upper bound.  A zero-initialised tail is an fp32 item with a host count. */
typedef struct {
  const float* dF; int32_t ldF; const float* anc_f32; const float* inv_norm; const int32_t* slot;
  int32_t n, C, plane; void* dfeat;
  int32_t dtype;
  const int32_t* n_rows_dev;
} mscs_scatter_item;
int mscs_scatter_sectors_batch(const mscs_scatter_item* items, int count, void* stream);
/* Channels-last feature maps (memory order [n][h][w][C]): an anchor is one contiguous row of C elements, so the gather
 * (+ L2 normalisation) and the scatter (normalisation backward into the pre-zeroed channels-last dense gradient) are
 * row copies driven by `pix` (global pixel id = image * plane + pixel of every sorted anchor row, -1 = not local).
 * `rows`: number of anchor rows, or their upper bound when `n_rows_dev` (device-resident count) is set.
 * `dtype` (last member, MSCS_DTYPE_*): element type of `feat` and `dfeat`. */
typedef struct {
  const void* feat; const int32_t* pix; const int32_t* n_rows_dev; int32_t rows, C;
  void* anc_bf16; float* anc_f32; float* inv_norm;          /* gather outputs / scatter inputs */
  const float* dF; int32_t ldF; void* dfeat;                /* scatter only */
  int32_t dtype;
} mscs_rows_item;
int mscs_gather_rows_nhwc_batch(const mscs_rows_item* items, int count, void* stream);
int mscs_scatter_rows_nhwc_batch(const mscs_rows_item* items, int count, void* stream);
/* Dense gradients of every scale written in ONE streaming pass, zeros included (no pre-zeroed buffer needed):
 * dF rows are first turned into dx rows IN PLACE (rows[s] rows of item s), then every 16 bytes of every dfeat are
 * written once (4 fp32 or 8 half pixels of a channel plane per store).  plane must be a multiple of 4 (fp32) or 8
 * (bf16 / fp16), dfeat 16-byte aligned. */
int mscs_scatter_dense_batch(const mscs_scatter_item* items, const int32_t* rows, int count, void* stream);

/* ---------------------------------------------------------------------------------------
 * One forward / one backward of the single-process path in ONE call each (csrc/step.cu): the same entry points as
 * above in the device-driven order, so that the host mirror crosses the ABI once per pass.  Replaces the host side
 * of DenseContrastiveLossV2_ms.forward's scale loop (_ms.py:44-82) and of its autograd backward.
 *
 * forward:  on `sample_stream` (ordered after what `main_stream` holds): workspace fills, mscs_sample_plan[_i16],
 *           mscs_plan_fetch_begin, mscs_sample_select_async;  on `main_stream` (ordered after the selection): the
 *           batched gather + normalisation, mscs_sim_forward;  then mscs_plan_fetch_end -- the one host wait.
 *           Returns like the parts (0 = ok; plan_host[s].error holds the reference's error conditions).
 *           sample_stream == main_stream runs everything on one stream.  plan_host == NULL: no plan fetch and no host
 *           wait -- the chain only enqueues work, and the sample stream joins back into main_stream (stream capture).
 * ------------------------------------------------------------------------------------- */
typedef struct {
  const mscs_sample_cfg* cfg;
  const void* labels;              /* int64 [n][H][W], or the int16 compact labels of mscs_label_pass (labels_i16 = 1) */
  int32_t labels_i16;
  int32_t v_cap;                   /* as mscs_sample_select_async */
  void* workspace;                 /* mscs_sample_workspace_bytes */
  mscs_scale_plan* plan_dev;       /* device plan records [num_scales] */
  const uint32_t* draws;           /* MT19937 / Philox stream buffer of this call */
  void* wait_event;                /* optional cudaEvent_t the sampling stream waits for (stream buffer complete) */
  int32_t* const* idx_ref; int32_t* const* pair_ref; int32_t* const* pix; int32_t* const* cls; int32_t* const* seg;
  int32_t* const* slot;            /* per scale, as mscs_sample_select_async */
  void* const* fill_ptrs; const int32_t* fill_values; const size_t* fill_bytes; int32_t n_fill;   /* mscs_fill_bytes */
  void* main_zero_ptr; size_t main_zero_bytes;   /* optional: cleared on main_stream while the sampling chain runs (the
                                      gradient-row accumulators of the backward) */
  int32_t gather_kind;             /* 0: NCHW (mscs_gather_item[num_scales]), 1: channels-last rows
                                      (mscs_rows_item[num_scales]) */
  const void* gather_items;
  const mscs_sim_job* job;         /* forward job (upper bounds + device-resident row counts) */
  void* stage_events[5];           /* optional cudaEvent_t, recorded at: sampling start / end (sample stream), gather
                                      start, gather end = similarity start, similarity end (main stream) */
} mscs_forward_chain_args;
int mscs_forward_chain(const mscs_forward_chain_args* args, void* sample_stream, void* main_stream,
                       mscs_scale_plan* plan_host);
/* backward: mscs_sim_backward, then mscs_scatter_dense_batch (count may be 0: no dense gradient wanted).
 * stage_events: NULL or 3 optional cudaEvent_t recorded before / between / after the two. */
int mscs_backward_chain(const mscs_sim_job* job, const float* grad_out, float* const* dF_sets, const int32_t* dF_ld,
                        const mscs_scatter_item* items, const int32_t* rows, int count, void* const* stage_events,
                        void* stream);

/* ---------------------------------------------------------------------------------------
 * Co-loss on the same label read (SURVEY.md 8f item 2).  The reference's LossWrapper evaluates a class-weighted
 * nn.CrossEntropyLoss(ignore_index, weight) on the full-resolution logits next to the contrastive loss
 * (losses/LossWrapper.py:22-31,81-82; TwoScaleLoss.py:62-73 applies it to two logit maps); both start from the int64
 * label map.
 *   mscs_label_pass    ONE sweep over the labels: compact int16 labels (-1 = outside [0, num_classes)) + the
 *                      full-resolution class histogram int32[num_classes] (zeroed inside).  The compact labels feed K1
 *                      (mscs_sample_hist_i16 / mscs_sample_plan_i16: same results as the int64 entry points) and the
 *                      CE kernels; the histogram gives the CE normaliser sum_valid w[y] before the logits are read.
 *   mscs_ce_forward    loss_and_denom[0] = sum_valid w[y] (logsumexp(x) - x_y) / denom,  [1] = denom = sum_c w[c] hist[c]
 *                      (c < K, c != ignore_index); logits NCHW (n, K, plane), plane % 4 == 0; weight NULL = ones;
 *                      labels >= K or == ignore_index are ignored; loss_sum_scratch: one double of device scratch.
 *   mscs_ce_backward   dlogits = (*grad_out / *denom) w[y] (softmax(x) - onehot(y)), zeros on ignored pixels: one fused
 *                      pass (ATen: log_softmax backward + nll_loss backward).
 *   `dtype` (MSCS_DTYPE_*): element type of logits and dlogits (fp32: 16-byte aligned, half: 8-byte aligned); the
 *   arithmetic is fp32 either way, dlogits are rounded to nearest even on store.
 * ------------------------------------------------------------------------------------- */
int mscs_label_pass(const int64_t* labels, int64_t n_pixels, int num_classes, int16_t* lab16, int32_t* hist,
                    void* stream);
int mscs_sample_hist_i16(const mscs_sample_cfg* cfg, const int16_t* lab16, void* workspace, void* stream);
int mscs_sample_plan_i16(const mscs_sample_cfg* cfg, const int16_t* lab16, void* workspace, mscs_scale_plan* plan_dev,
                         void* stream);
int mscs_ce_forward(const void* logits, const int16_t* lab16, int n, int K, int plane, const float* weight,
                    int ignore_index, const int32_t* hist, int num_classes, double* loss_sum_scratch,
                    float* loss_and_denom, void* stream, int dtype);
int mscs_ce_backward(const void* logits, const int16_t* lab16, int n, int K, int plane, const float* weight,
                     int ignore_index, const float* grad_out, const float* denom, void* dlogits, void* stream,
                     int dtype);

/* ---------------------------------------------------------------------------------------
 * Projector tail on the sampled rows only (SURVEY.md 8f item 1; models/Projector.py:49-72: the projector ends in
 * nn.Conv2d(c_prev, d, kernel_size=1), evaluated densely by the reference although the loss reads <= 10k pixels per
 * scale).  The 1x1 convolution of the sampled pixels is a plain (N x c_prev) x (c_prev x d) GEMM on the host side's
 * library of choice; these calls move the rows, every scale in one launch per element type of the maps.  The rows are
 * fp32 (N x C, row stride C) and not normalised: a half map gives the same rows as its exact fp32 widening.
 *   mscs_gather_raw_batch       NCHW: rows[slot[b*plane+p]][:] = feat[b, :, p], in the address order of the slot map
 *                               (mscs_gather_item: `anc_f32` receives the rows; anc_bf16, inv_norm and n_rows_dev are
 *                               not used -- the slot map holds the sampled rows only; plane % 8 == 0)
 *   mscs_gather_raw_rows_batch  channels-last: rows[r][:] = feat[pix[r]][:] for r below the count (mscs_rows_item:
 *                               `anc_f32` receives the rows, `rows` / `n_rows_dev` as for mscs_gather_rows_nhwc_batch)
 * The way back is the dense writers above: an item of mscs_scatter_dense_batch or mscs_scatter_rows_nhwc_batch whose
 * anc_f32 and inv_norm are both NULL stores its rows dF as they are (no normalisation backward); exactly one of the two
 * being NULL is rejected.
 * ------------------------------------------------------------------------------------- */
int mscs_gather_raw_batch(const mscs_gather_item* items, int count, void* stream);
int mscs_gather_raw_rows_batch(const mscs_rows_item* items, int count, void* stream);

/* ---------------------------------------------------------------------------------------
 * Pooled cross-batch mode -- the exchange between the GPUs of one box over NVLink peer memory.  (Not a reference
 * behaviour: the reference evaluates the loss per rank, utils/distributed.py:63-73 `concat_all_gather` is imported by
 * DenseContrastiveLossV2_ms.py:3 and never called; BASELINE.json's north_star adds this configuration.)
 * Every rank owns one exchange slab with the SAME layout; `slabs[r]` is rank r's slab as mapped into this process
 * (slabs[rank] = the local allocation).  Word r of the first 32 bytes of a slab is the barrier epoch of rank r.
 * ------------------------------------------------------------------------------------- */
/* cudaMalloc + zero fill + CUDA IPC export (handle_out: MSCS_IPC_HANDLE_BYTES bytes, to be sent to the peers) */
int mscs_xchg_alloc(size_t bytes, void** dev_ptr, unsigned char* handle_out);
/* map a peer's slab from its IPC handle (peer access is enabled on first use) / unmap it */
int mscs_xchg_open(const unsigned char* handle, void** dev_ptr);
int mscs_xchg_close(void* dev_ptr);
int mscs_xchg_free(void* dev_ptr);
/* Device-side barrier across the ranks (async, one tiny kernel): everything this rank enqueued on `stream` before the
 * call -- peer stores included -- is visible to every rank after ITS barrier call with the same epoch has completed.
 * `epoch`: strictly increasing per slab (1, 2, 3, ...), the same sequence on every rank.  A rank that waits longer than
 * timeout_s seconds (<= 0: 20 s) traps, i.e. the stream reports a launch failure instead of hanging. */
int mscs_xchg_barrier(void* const* slabs, int world, int rank, uint32_t epoch, double timeout_s, void* stream);
/* copy `count` (<= 48) float ranges src[src_float_off[j] .. + len[j]) (private memory of this rank: the row statistics
 * of its anchor rows, accumulated by the sweeps) to float offset float_off[j] of EVERY rank's slab, its own included */
int mscs_xchg_push(void* const* slabs, int world, const float* src, const int64_t* src_float_off,
                   const int64_t* float_off, const int32_t* len, int count, void* stream);
/* K2 fused with the all-gather of the normalised key set: as mscs_gather_normalize_sectors, but every bf16 anchor row
 * is stored into the operand matrix at byte offset bf16_byte_off of EVERY rank's slab (same sorted row everywhere: the
 * plan is global); fp32 rows and inverse norms stay local.  Also zeroes the local padding rows [N, N_pad). */
int mscs_gather_normalize_p2p(const float* feat, int n, int C, int plane, const int32_t* slot, int N,
                              const int32_t* n_rows_dev /* optional: N read on the device, e.g. &plan_dev[s].N */,
                              void* const* slabs, int world, int rank, size_t bf16_byte_off, float* anc_f32,
                              float* inv_norm, void* stream);
/* as mscs_scatter_sectors, with gradient row i read from rank (i / rows_per_rank)'s slab at dF_byte_off (the rank
 * that computed it: anchor rows are sharded in 128-aligned blocks of rows_per_rank rows) */
int mscs_scatter_sectors_pull(void* const* slabs, int world, size_t dF_byte_off, int rows_per_rank, int ldF,
                              const float* anc_f32, const float* inv_norm, const int32_t* slot, int n, int C, int plane,
                              float* dfeat, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MSCS_H_ */
