"""ctypes binding of libmscs.so (include/mscs.h).  No fallback: if the library is missing or a
call fails, a RuntimeError is raised -- there is no CPU or PyTorch path behind this module."""
import ctypes as C
import os

MAX_SCALES, MAX_TERMS = 8, 16
MAX_RANKS, IPC_HANDLE_BYTES = 8, 64      # MSCS_MAX_RANKS, MSCS_IPC_HANDLE_BYTES
DTYPE_F32, DTYPE_BF16, DTYPE_F16 = 0, 1, 2   # MSCS_DTYPE_*: element type of feature maps / logits and their gradients

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MSCS_LIB") or os.path.join(_HERE, "libmscs.so")   # MSCS_LIB: profiling build


class SampleCfg(C.Structure):
    _fields_ = [("n", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("num_scales", C.c_int32),
                ("fh", C.c_int32 * MAX_SCALES), ("fw", C.c_int32 * MAX_SCALES),
                ("num_classes", C.c_int32), ("min_views", C.c_int32), ("max_views", C.c_int32),
                ("max_total", C.c_int32), ("n_global", C.c_int32), ("image_base", C.c_int32)]


class ScalePlan(C.Structure):
    _fields_ = [("T", C.c_int32), ("V", C.c_int32), ("N", C.c_int32), ("min_count", C.c_int32),
                ("log_flag", C.c_int32), ("dl_h", C.c_int32), ("dl_w", C.c_int32), ("error", C.c_int32),
                ("draw_base", C.c_int64), ("draws", C.c_int64)]


class GatherItem(C.Structure):
    _fields_ = [("feat", C.c_void_p), ("n", C.c_int32), ("C", C.c_int32), ("plane", C.c_int32), ("slot", C.c_void_p),
                ("n_rows_dev", C.c_void_p), ("anc_bf16", C.c_void_p), ("anc_f32", C.c_void_p), ("inv_norm", C.c_void_p),
                ("dtype", C.c_int32)]


class ScatterItem(C.Structure):
    _fields_ = [("dF", C.c_void_p), ("ldF", C.c_int32), ("anc_f32", C.c_void_p), ("inv_norm", C.c_void_p),
                ("slot", C.c_void_p), ("n", C.c_int32), ("C", C.c_int32), ("plane", C.c_int32), ("dfeat", C.c_void_p),
                ("dtype", C.c_int32), ("n_rows_dev", C.c_void_p)]


class RowsItem(C.Structure):
    _fields_ = [("feat", C.c_void_p), ("pix", C.c_void_p), ("n_rows_dev", C.c_void_p), ("rows", C.c_int32),
                ("C", C.c_int32), ("anc_bf16", C.c_void_p), ("anc_f32", C.c_void_p), ("inv_norm", C.c_void_p),
                ("dF", C.c_void_p), ("ldF", C.c_int32), ("dfeat", C.c_void_p), ("dtype", C.c_int32)]


class Term(C.Structure):
    _fields_ = [("a_bf16", C.c_void_p), ("k_bf16", C.c_void_p),
                ("a_cls", C.c_void_p), ("k_seg", C.c_void_p), ("k_cls", C.c_void_p), ("a_seg", C.c_void_p),
                ("N1", C.c_int32), ("N2", C.c_int32), ("self_mask", C.c_int32), ("need_dk", C.c_int32),
                ("temperature", C.c_float), ("weight", C.c_float), ("a_set", C.c_int32), ("k_set", C.c_int32),
                ("row_begin", C.c_int32), ("row_end", C.c_int32), ("krow_begin", C.c_int32), ("krow_end", C.c_int32),
                ("neg_sum", C.c_void_p), ("pos_sum", C.c_void_p), ("s_sum", C.c_void_p),
                ("coef_s", C.c_void_p), ("coef_pn", C.c_void_p), ("n1_dev", C.c_void_p), ("n2_dev", C.c_void_p)]


class SimJob(C.Structure):
    _fields_ = [("num_terms", C.c_int32), ("C_pad", C.c_int32), ("num_classes", C.c_int32),
                ("terms", Term * MAX_TERMS), ("term_loss", C.c_void_p), ("total_loss", C.c_void_p),
                ("work", C.c_void_p), ("total_out", C.c_void_p)]


class ForwardChainArgs(C.Structure):
    """mscs_forward_chain_args (include/mscs.h)."""
    _fields_ = [("cfg", C.c_void_p), ("labels", C.c_void_p), ("labels_i16", C.c_int32), ("v_cap", C.c_int32),
                ("workspace", C.c_void_p), ("plan_dev", C.c_void_p), ("draws", C.c_void_p), ("wait_event", C.c_void_p),
                ("idx_ref", C.c_void_p), ("pair_ref", C.c_void_p), ("pix", C.c_void_p), ("cls", C.c_void_p),
                ("seg", C.c_void_p), ("slot", C.c_void_p),
                ("fill_ptrs", C.c_void_p), ("fill_values", C.c_void_p), ("fill_bytes", C.c_void_p), ("n_fill", C.c_int32),
                ("main_zero_ptr", C.c_void_p), ("main_zero_bytes", C.c_size_t),
                ("gather_kind", C.c_int32), ("gather_items", C.c_void_p), ("job", C.c_void_p),
                ("stage_events", C.c_void_p * 5)]


_PTRS = C.POINTER(C.c_void_p)
_SIGNATURES = {
    "mscs_version": (C.c_char_p, []),
    "mscs_last_error": (C.c_char_p, []),
    "mscs_device_ok": (C.c_int, []),
    "mscs_read_to_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "mscs_fill_bytes": (C.c_int, [_PTRS, C.POINTER(C.c_int32), C.POINTER(C.c_size_t), C.c_int, C.c_void_p]),
    "mscs_debug_trap_info": (C.c_int, [C.c_char_p, C.c_int]),
    "mscs_debug_wait_profile_fwd": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mscs_debug_wait_profile_bwd": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mscs_debug_trace_bwd": (C.c_int, [C.c_void_p, C.c_int]),
    "mscs_debug_trace_fwd": (C.c_int, [C.c_void_p, C.c_int]),
    "mscs_debug_fwd_timeline": (C.c_int, [C.c_void_p, C.c_int]),
    "mscs_debug_cta_spans_fwd": (C.c_int, [C.c_void_p, C.c_int]),
    "mscs_sample_workspace_bytes": (C.c_size_t, [C.POINTER(SampleCfg)]),
    "mscs_sample_max_draws": (C.c_size_t, [C.POINTER(SampleCfg)]),
    "mscs_sample_plan": (C.c_int, [C.POINTER(SampleCfg), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mscs_sample_counts_offset": (C.c_size_t, [C.POINTER(SampleCfg), C.c_int]),
    "mscs_sample_hist": (C.c_int, [C.POINTER(SampleCfg), C.c_void_p, C.c_void_p, C.c_void_p]),
    "mscs_sample_plan_from_counts": (C.c_int, [C.POINTER(SampleCfg), _PTRS, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mscs_plan_fetch": (C.c_int, [C.c_void_p, C.POINTER(ScalePlan), C.c_int, C.c_void_p]),
    "mscs_plan_fetch_begin": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "mscs_plan_fetch_end": (C.c_int, [C.POINTER(ScalePlan), C.c_int]),
    "mscs_sample_select_async": (C.c_int, [C.POINTER(SampleCfg), C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                           _PTRS, _PTRS, _PTRS, _PTRS, _PTRS, _PTRS, C.c_void_p]),
    "mscs_gather_normalize_sectors_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "mscs_scatter_sectors_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "mscs_gather_rows_nhwc_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "mscs_scatter_rows_nhwc_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "mscs_scatter_dense_batch": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.c_int, C.c_void_p]),
    "mscs_mt19937_stream": (C.c_int, [C.c_void_p, C.c_int, C.c_uint64, C.c_void_p, C.c_void_p]),
    "mscs_philox_stream": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p]),
    "mscs_philox_stream_dev": (C.c_int, [C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "mscs_sample_select": (C.c_int, [C.POINTER(SampleCfg), C.POINTER(ScalePlan), C.c_void_p, C.c_void_p,
                                     _PTRS, _PTRS, _PTRS, _PTRS, _PTRS, _PTRS, C.c_void_p]),
    "mscs_mt19937_advance_host": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.c_uint64]),
    "mscs_gather_normalize": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p]),
    "mscs_sim_workspace_bytes": (C.c_size_t, [C.POINTER(SimJob)]),
    "mscs_sim_forward": (C.c_int, [C.POINTER(SimJob), C.c_void_p]),
    "mscs_forward_chain": (C.c_int, [C.POINTER(ForwardChainArgs), C.c_void_p, C.c_void_p, C.c_void_p]),
    "mscs_backward_chain": (C.c_int, [C.POINTER(SimJob), C.c_void_p, _PTRS, C.POINTER(C.c_int32), C.c_void_p,
                                      C.POINTER(C.c_int32), C.c_int, _PTRS, C.c_void_p]),
    "mscs_sim_forward_sweeps": (C.c_int, [C.POINTER(SimJob), C.c_void_p]),
    "mscs_sim_finalize": (C.c_int, [C.POINTER(SimJob), C.c_void_p]),
    "mscs_sim_backward": (C.c_int, [C.POINTER(SimJob), C.c_void_p, _PTRS, C.POINTER(C.c_int32), C.c_void_p]),
    "mscs_sim_backward_sets": (C.c_int, [C.POINTER(SimJob), C.c_void_p, _PTRS, C.POINTER(C.c_int32), C.c_uint32,
                                         C.c_void_p]),
    "mscs_debug_sim_forward_simt": (C.c_int, [C.POINTER(SimJob), _PTRS, C.c_void_p]),
    "mscs_debug_sim_backward_simt": (C.c_int, [C.POINTER(SimJob), _PTRS, C.c_void_p, _PTRS, C.POINTER(C.c_int32),
                                               C.c_void_p]),
    "mscs_scatter_grad": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                    C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "mscs_label_pass": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mscs_sample_hist_i16": (C.c_int, [C.POINTER(SampleCfg), C.c_void_p, C.c_void_p, C.c_void_p]),
    "mscs_sample_plan_i16": (C.c_int, [C.POINTER(SampleCfg), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mscs_ce_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                  C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "mscs_ce_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "mscs_gather_raw_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "mscs_gather_raw_rows_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "mscs_xchg_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p), C.c_char_p]),
    "mscs_xchg_open": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "mscs_xchg_close": (C.c_int, [C.c_void_p]),
    "mscs_xchg_free": (C.c_int, [C.c_void_p]),
    "mscs_xchg_barrier": (C.c_int, [_PTRS, C.c_int, C.c_int, C.c_uint32, C.c_double, C.c_void_p]),
    "mscs_xchg_push": (C.c_int, [_PTRS, C.c_int, C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                 C.POINTER(C.c_int32), C.c_int, C.c_void_p]),
    "mscs_gather_normalize_p2p": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, _PTRS,
                                            C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "mscs_scatter_sectors_pull": (C.c_int, [_PTRS, C.c_int, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "mscs_gather_rows_p2p": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, _PTRS, C.c_int, C.c_int,
                                       C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "mscs_scatter_rows_pull": (C.c_int, [_PTRS, C.c_int, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "mscs_local_rows_batch": (C.c_int, [_PTRS, _PTRS, C.POINTER(C.c_int32), _PTRS, _PTRS, _PTRS, C.c_void_p, C.c_int,
                                        C.c_void_p]),
}
EXPORTS = tuple(_SIGNATURES)

_lib = None


def load():
    """Load libmscs.so (once).  Raises RuntimeError when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; "
                               f"g.build()'` (or `make -C {os.path.join(_HERE, 'csrc')}`). There is no fallback path.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def trap_info():
    buf = C.create_string_buffer(4096)
    n = load().mscs_debug_trap_info(buf, 4096)
    return buf.value.decode() if n > 0 else ""


def check(rc, what):
    if rc != 0:
        msg = load().mscs_last_error().decode()
        raise RuntimeError(f"{what} failed (code {rc}): {msg} {trap_info()}")


def ptr_array(ptrs):
    arr = (C.c_void_p * len(ptrs))(*ptrs)
    return arr
