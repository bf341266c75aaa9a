// sim_tc.cuh -- pieces shared by the tcgen05 forward and backward kernels: the work table
// (balanced contiguous tile ranges per CTA), the TMA tensor-map factory, shared-memory carving.
#pragma once
#include "ptx.cuh"
#include "sim_common.cuh"

namespace mscs {

constexpr int kTileN = 128;          // key rows (logit columns) per tile
constexpr int kKBlk = 64;            // bf16 elements per 128-byte swizzled row
constexpr int kBlkBytes = 128 * 128; // one [128 rows][64 bf16] operand block = 16 KB

// one unit of work = one (row block, column tile); an item is a run of column tiles of one row block
struct WorkItem { int owner, rb, ct0, ct1; };
// `pad`: virtual units charged to every item on top of its tiles when the work is cut into equal shares -- the
// fixed cost of starting a run (operand load, pipeline fill, accumulator flush), in tiles.  A CTA whose share is
// made of many short runs then gets fewer tiles instead of finishing late (sim_bwd: 17% tail before).
struct WorkTable { const WorkItem* items; const int* prefix; int nitems; int pad; };

struct Segment { int owner, rb, c_begin, c_end; };

struct Walker {
  const WorkTable& w;
  int u, u_end, item;
  __device__ Walker(const WorkTable& wt) : w(wt) {
    const long long total = wt.prefix[wt.nitems];
    u = (int)(total * blockIdx.x / gridDim.x);
    u_end = (int)(total * (blockIdx.x + 1) / gridDim.x);
    int lo = 0, hi = wt.nitems;        // largest item with prefix[item] <= u
    while (lo < hi) {
      int mid = (lo + hi + 1) >> 1;
      if (wt.prefix[mid] <= u) lo = mid; else hi = mid - 1;
    }
    item = lo;
  }
  // prefix[] counts pad + tiles per item (items without tiles count 0); the first `pad` virtual units of an
  // item are its start-up charge and map to no tile
  __device__ bool next(Segment& s) {
    while (u < u_end) {
      while (w.prefix[item + 1] <= u) ++item;
      const WorkItem it = w.items[item];
      const int base = w.prefix[item];
      const int e = min(u_end, w.prefix[item + 1]);
      const int b0 = max(0, u - base - w.pad), b1 = max(0, e - base - w.pad);
      u = e;
      if (b1 > b0) {
        s.owner = it.owner; s.rb = it.rb;
        s.c_begin = it.ct0 + b0;
        s.c_end = it.ct0 + b1;
        return true;
      }
    }
    return false;
  }
};

// work-table builder (sim_fwd.cu): one item per (owner, row block)
// n1_dev / n2_dev: optional device-resident row counts (then N1 / N2 are upper bounds, see mscs_term)
struct BuildTerm { const int* a_cls; const int* k_seg; int N1, N2, item_base, blk_lo, ct_lo, ct_hi;
                   const int* n1_dev; const int* n2_dev; };
struct BuildArgs { BuildTerm t[MSCS_MAX_PASSES]; int num_terms, nitems, rows_per_item, mode, pad; WorkItem* items; int* prefix;
                   WorkItem* items1; int* prefix1; };   // items1 / prefix1 non-null: a second block builds the mode + 1 table
int launch_build_work(const BuildArgs& b, cudaStream_t st);
int trap_buffer_device_ptr(unsigned long long** out);
// each translation unit with tensor kernels installs the buffer into its own g_trap_buf copy
static inline int ensure_trap_buffer() {
  static bool done = false;
  if (done) return 0;
  unsigned long long* d = nullptr;
  if (int rc = trap_buffer_device_ptr(&d)) return rc;
  MSCS_CUDA(cudaMemcpyToSymbol(ptx::g_trap_buf, &d, sizeof(d)));
  done = true;
  return 0;
}
int sm_count();
int persistent_ctas();   // grid of the persistent tensor kernels (SM count minus the spare SMs, sim_fwd.cu)

// TMA tensor map for a row-major (rows, C_pad) bf16 matrix, box = {64 elements, 128 rows}, 128B swizzle
int make_tensor_map(CUtensorMap* out, const void* base, int rows, int c_pad);

}  // namespace mscs
