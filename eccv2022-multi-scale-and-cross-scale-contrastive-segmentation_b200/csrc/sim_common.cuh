// sim_common.cuh -- term / pass descriptors shared by the similarity kernels.
//
// Loss maths (SURVEY.md Appendix A; V2.py:173-188, _ms.py:132-156), rows i = anchors,
// columns j = keys, l_ij = a_i.k_j / tau, E_ij = exp(l_ij):
//   neg_i = sum_{y_j != y_i} E_ij
//   pos_i = sum_{j in P_i} [ l_ij - log(E_ij + neg_i) ]      P_i: y_j == y_i (and j != i if self)
//   S_i   = sum_{j in P_i} 1 / (E_ij + neg_i)
//   loss  = mean_i ( -pos_i / div_i ),  div_i = |P_i| (self) or max(|P_i|, 1) (cross-scale)
// backward, with c_i = 1/(div_i N1):
//   G_ij = -c_i neg_i / (E_ij + neg_i)   (positive)      G_ij = c_i S_i E_ij   (negative)
//   dA = G K / tau,  dK = G^T A / tau;  single-scale: dF = (G + G^T) F / tau.
// Rows of every anchor set are sorted by class, so the positives of row i are the contiguous
// key rows [k_seg[y_i], k_seg[y_i + 1]).
#pragma once
#include "common.cuh"

namespace mscs {

constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

// one backward pass: dX_rows += scale * W(rows, cols) * Y_cols
struct BwdPass {
  const void* x_bf16; const void* y_bf16;     // rows / cols operand matrices (N_pad, C_pad) bf16
  const int* row_cls; const int* col_seg;     // class of each row; class segments of the column set
  const int* col_cls;                         // class of each column (SIMT validation kernels)
  const float* row_cs; const float* row_cpn; const float* row_neg;   // row-side coefficients or null
  const float* col_cs; const float* col_cpn; const float* col_neg;   // col-side coefficients or null
  int n_rows, n_cols;
  const int* n_rows_dev; const int* n_cols_dev;   // device-resident counts (n_rows / n_cols: upper bounds) or null
  int rb_lo, rb_hi;       // row tiles (128 rows) this rank handles
  int self_mask;
  int row_set, col_set;
  float scale_log2;      // log2(e)/tau
  float out_scale;       // weight / tau  (times *grad_out on the device)
};

static inline int build_passes(const mscs_sim_job* job, BwdPass* out) {
  int np = 0;
  for (int t = 0; t < job->num_terms; ++t) {
    const mscs_term& m = job->terms[t];
    BwdPass p{};
    p.x_bf16 = m.a_bf16; p.y_bf16 = m.k_bf16; p.row_cls = m.a_cls; p.col_seg = m.k_seg; p.col_cls = m.k_cls;
    p.row_cs = m.coef_s; p.row_cpn = m.coef_pn; p.row_neg = m.neg_sum;
    p.n_rows = m.N1; p.n_cols = m.N2; p.self_mask = m.self_mask; p.row_set = m.a_set; p.col_set = m.k_set;
    p.n_rows_dev = m.n1_dev; p.n_cols_dev = m.n2_dev;
    p.scale_log2 = kLog2e / m.temperature; p.out_scale = m.weight / m.temperature;
    { const bool all = m.row_begin == 0 && m.row_end == 0;      // 0,0 = every row; begin == end = none
      p.rb_lo = (all ? 0 : m.row_begin) / 128; p.rb_hi = ((all ? m.N1 : m.row_end) + 127) / 128;
      if (!all && m.row_end == m.row_begin) p.rb_hi = p.rb_lo; }
    if (m.self_mask) { p.col_cs = m.coef_s; p.col_cpn = m.coef_pn; p.col_neg = m.neg_sum; }
    out[np++] = p;
    if (!m.self_mask && m.need_dk) {
      BwdPass q{};
      q.x_bf16 = m.k_bf16; q.y_bf16 = m.a_bf16; q.row_cls = m.k_cls; q.col_seg = m.a_seg; q.col_cls = m.a_cls;
      q.col_cs = m.coef_s; q.col_cpn = m.coef_pn; q.col_neg = m.neg_sum;
      q.n_rows = m.N2; q.n_cols = m.N1; q.self_mask = 0; q.row_set = m.k_set; q.col_set = m.a_set;
      q.n_rows_dev = m.n2_dev; q.n_cols_dev = m.n1_dev;
      q.scale_log2 = p.scale_log2; q.out_scale = p.out_scale;
      { const bool all = m.krow_begin == 0 && m.krow_end == 0;
        q.rb_lo = (all ? 0 : m.krow_begin) / 128; q.rb_hi = ((all ? m.N2 : m.krow_end) + 127) / 128;
        if (!all && m.krow_end == m.krow_begin) q.rb_hi = q.rb_lo; }
      out[np++] = q;
    }
  }
  return np;
}

static inline int validate_job(const mscs_sim_job* job) {
  MSCS_CHECK_ARG(job != nullptr, "job is null");
  MSCS_CHECK_ARG(job->num_terms >= 1 && job->num_terms <= MSCS_MAX_TERMS, "num_terms %d out of range",
                 job->num_terms);
  MSCS_CHECK_ARG(job->C_pad >= 64 && job->C_pad <= 256 && job->C_pad % 64 == 0, "C_pad %d unsupported",
                 job->C_pad);
  MSCS_CHECK_ARG(job->term_loss && job->total_loss, "null output pointer");
  for (int t = 0; t < job->num_terms; ++t) {
    const mscs_term& m = job->terms[t];
    MSCS_CHECK_ARG(m.a_bf16 && m.k_bf16 && m.a_cls && m.k_seg && m.k_cls && m.a_seg, "term %d: null input", t);
    MSCS_CHECK_ARG(m.neg_sum && m.pos_sum && m.s_sum && m.coef_s && m.coef_pn, "term %d: null stats", t);
    MSCS_CHECK_ARG(m.N1 >= 1 && m.N2 >= 1, "term %d: empty", t);
    MSCS_CHECK_ARG(m.temperature > 0.f, "term %d: temperature must be positive", t);
    MSCS_CHECK_ARG(!m.self_mask || (m.a_bf16 == m.k_bf16 && m.N1 == m.N2), "term %d: self term needs a == k", t);
    MSCS_CHECK_ARG(m.row_begin >= 0 && m.row_begin <= m.row_end && m.row_end <= m.N1 &&
                   (m.row_begin % 128 == 0 || m.row_begin == m.N1) && (m.row_end % 128 == 0 || m.row_end == m.N1),
                   "term %d: bad anchor row range [%d,%d)", t, m.row_begin, m.row_end);
    MSCS_CHECK_ARG(m.krow_begin >= 0 && m.krow_begin <= m.krow_end && m.krow_end <= m.N2 &&
                   (m.krow_begin % 128 == 0 || m.krow_begin == m.N2) && (m.krow_end % 128 == 0 || m.krow_end == m.N2),
                   "term %d: bad key row range [%d,%d)", t, m.krow_begin, m.krow_end);
    MSCS_CHECK_ARG(m.a_set >= 0 && m.a_set < MSCS_MAX_SCALES && m.k_set >= 0 && m.k_set < MSCS_MAX_SCALES,
                   "term %d: bad set index", t);
  }
  return 0;
}

// launched by both implementations after the two forward sweeps
// zero_acc: the caller did not run k_row_ranges (which clears the accumulators) on this job->work before
int launch_finalize(const mscs_sim_job* job, cudaStream_t st, bool zero_acc = false);

}  // namespace mscs
