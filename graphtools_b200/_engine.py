"""ctypes binding of libgtb200.so (the C ABI declared in include/gtb200.h).

PyTorch is used for device memory and streams only; every compute step is a call into the
hand-written sm_100a kernels.  There is NO CPU fallback: importing the engine without the built
library, or calling it without a CUDA device, raises.
"""
import ctypes
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
# GTB_LIB points the binding at another build of the same ABI (kernel experiments); default = the in-tree library
LIB_PATH = os.environ.get("GTB_LIB") or os.path.join(_HERE, "libgtb200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "gtb200.h")

_lib = None
launch_count = 0  # number of C-ABI compute calls issued (each launches >= 1 kernel)
kernel_launches = 0  # kernels launched by those calls (bench.py reports this)

c_void_p, c_int, c_int64, c_double, c_float = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int64,
                                                ctypes.c_double, ctypes.c_float)

# name -> (argtypes, kernels launched per call)
_P = c_void_p
_SIGS = {
    "gtb_col_mean": ([_P, c_int64, c_int, _P, _P, _P], 2),
    "gtb_prepare_operand": ([_P, c_int64, c_int, _P, _P, c_int64, c_int, _P, _P, _P], 2),
    "gtb_gather_operand": ([_P, c_int64, _P, _P, c_int64, _P, c_int64, c_int, _P, _P], 1),
    "gtb_knn_topk_simt": ([_P, _P, c_int64, c_int64, _P, _P, c_int64, c_int64, c_int, c_int, _P, _P, _P], 1),
    "gtb_knn_radius_simt": ([_P, _P, _P, c_int64, c_int64, _P, _P, c_int64, c_int64, c_int, _P, c_int64, _P, _P,
                             _P], 1),
    "gtb_row_norms": ([_P, c_int64, c_int, _P, c_int64, _P, _P, _P], 1),
    "gtb_prepare_operand_tc": ([_P, c_int64, c_int, _P, c_int, _P, _P, c_int64, c_int, c_int, c_float, _P, _P, _P], 2),
    "gtb_split_operand_tc": ([_P, c_int64, c_int, _P, c_int, _P, _P, c_int64, c_int, c_int, c_float, _P, _P], 1),
    "gtb_knn_topk_tc": ([_P, _P, _P, c_int64, c_int64, _P, _P, c_int64, c_int64, c_int, c_int, c_int, c_int, c_int, _P,
                         _P, _P, _P, _P], 1),
    "gtb_knn_topk_tc_seeded": ([_P, _P, _P, c_int64, c_int64, _P, _P, c_int64, c_int64, c_int, c_int, c_int, c_int, c_int,
                                _P, c_int, _P, _P, _P, _P, _P, _P, _P, _P], 1),
    "gtb_knn_seed_tc": ([_P, _P, c_int64, c_int64, _P, c_int64, c_int64, c_int, c_int, c_int, _P, _P, _P], 1),
    "gtb_order_assign": ([_P, c_int64, c_int, c_int, _P, _P], 1),
    "gtb_order_sort": ([_P, c_int64, c_int, _P, _P, _P], 3),
    "gtb_tile_geometry": ([_P, c_int64, c_int, c_int, _P, c_int64, c_int64, _P, _P, _P], 1),
    "gtb_tile_lists_count": ([_P, _P, _P, c_int64, _P, _P, c_int64, c_int, _P, _P, _P], 1),
    "gtb_tile_lists_fill": ([_P, c_int64, c_int64, _P, _P, _P], 1),
    "gtb_unpermute_candidates": ([_P, _P, c_int64, c_int, c_int, _P, _P, _P, _P, _P], 1),
    "gtb_knn_radius_tc": ([_P, _P, _P, _P, c_int64, c_int64, _P, _P, c_int64, c_int64, c_int, c_int, c_int, _P, c_int64,
                           _P, _P, _P, _P], 1),
    "gtb_knn_count_tc": ([_P, _P, _P, _P, c_int64, c_int64, _P, _P, c_int64, c_int64, c_int, c_int, c_int, c_int, c_int,
                          c_int, _P, _P, _P], 1),
    "gtb_knn_count_simt": ([_P, _P, _P, c_int64, c_int64, _P, _P, c_int64, c_int64, c_int, c_int, c_int, c_int, _P, _P],
                           1),
    "gtb_knn_count_bound": ([_P, _P, c_int64, c_int64, c_int, c_int, c_float, _P, c_float, c_double, c_int, c_int,
                             c_int64, c_double, c_double, _P, c_int, c_double, _P, _P, _P, _P, _P], 1),
    "gtb_refine_topk": ([_P, c_int64, _P, c_int, c_int, _P, c_int, c_int, _P, c_int, _P, c_float, c_double, c_int, c_int64, c_double,
                         c_double, _P, c_int, c_double, _P, _P, _P, _P, _P, _P, _P, _P], 1),
    "gtb_compact_todo": ([_P, c_int64, _P, _P, _P], 1),
    "gtb_scatter_pairs": ([_P, c_int64, _P, _P, c_int64, _P, _P], 1),
    "gtb_refine_ball": ([_P, _P, _P, c_int64, _P, c_int, c_int, _P, _P, _P, c_int, c_int64, c_double, c_double, _P, c_int,
                         c_double, _P, _P, _P, _P, _P, c_int, _P], 2),
    "gtb_csr_gather": ([_P, _P, _P, _P, _P, c_int64, c_int, _P, c_int64, _P, _P, _P, _P, _P, _P, _P], 2),
    "gtb_exclusive_scan": ([_P, c_int64, _P, _P, _P], 1),
    "gtb_cast_indptr": ([_P, c_int64, _P, _P], 1),
    "gtb_transpose_count": ([_P, c_int64, c_int, _P, c_int64, _P], 1),
    "gtb_transpose_scatter": ([_P, _P, _P, c_int64, c_int, c_int, _P, _P, _P], 1),
    "gtb_csr_sort_rows": ([_P, _P, _P, c_int64, _P, _P], 2),
    "gtb_rec_sort_rows": ([_P, _P, c_int64, _P, c_int, _P, _P], 2),
    "gtb_records_count": ([_P, c_int64, c_int, _P, c_int64, _P], 1),
    "gtb_records_scatter": ([_P, c_int64, c_int, _P, _P, _P], 1),
    "gtb_sym_merge_count": ([_P, _P, _P, _P, _P, c_int64, c_int, c_double, _P, _P, _P], 2),
    "gtb_sym_merge_fill": ([_P, _P, _P, _P, _P, c_int64, c_int, c_int, c_double, _P, _P, _P, _P, _P, _P, _P], 1),
    "gtb_asym_check": ([_P, _P, _P, c_int64, _P, _P], 1),
    "gtb_row_finalize": ([_P, _P, _P, c_int64, _P, _P, _P, c_int, _P], 1),
    "gtb_anisotropy": ([_P, _P, _P, _P, c_double, c_int64, _P], 1),
    "gtb_route_count": ([_P, _P, c_int64, c_int, c_int, _P, _P], 1),
    "gtb_route_fill": ([_P, _P, _P, c_int64, c_int, c_int, c_int, _P, _P, _P, _P], 1),
    "gtb_csr_to_dense": ([_P, _P, _P, c_int64, c_int64, _P, _P], 1),
    "gtb_block_count": ([_P, c_int64, _P, _P, _P], 1),
    "gtb_block_fill": ([_P, _P, _P, c_int64, _P, _P, _P, _P, c_double, _P, _P, _P, _P, _P], 1),
    "gtb_cluster_aggregate_count": ([_P, _P, _P, c_int64, _P, c_int, _P, _P, _P], 2),
    "gtb_cluster_aggregate_fill": ([_P, _P, _P, c_int64, _P, _P, _P, _P, _P, _P, _P, c_int, _P, _P], 3),
    "gtb_landmark_op": ([_P, _P, _P, _P, _P, c_int64, c_int, _P, _P, _P], 2),
    "gtb_dense_kernel": ([_P, c_int64, _P, c_int64, c_int, c_int, c_int, c_int, _P, _P, c_double, c_double, c_int,
                          c_double, _P, _P, _P], 1),
    "gtb_knn_topk_simt_l1": ([_P, c_int64, c_int64, _P, c_int64, c_int64, c_int, c_int, _P, _P, _P], 1),
    "gtb_knn_radius_simt_l1": ([_P, _P, c_int64, c_int64, _P, c_int64, c_int64, c_int, _P, c_int64, _P, _P, _P], 1),
    "gtb_dense_row_scale": ([_P, _P, c_int64, c_int64, _P, _P], 1),
    "gtb_dense_anisotropy": ([_P, _P, c_double, c_int64, _P, _P], 1),
    "gtb_dense_rowsum": ([_P, c_int64, c_int64, _P, _P], 1),
    "gtb_spmm_csr": ([_P, _P, _P, c_int64, _P, c_int64, c_int, _P, c_int64, _P], 1),
    "gtb_spmm_cheb": ([_P, _P, _P, c_int64, _P, c_int64, c_int, c_double, c_double, c_double, _P, c_int64, _P, c_int64,
                       _P], 1),
    "gtb_spmm_cheb_acc": ([_P, _P, _P, c_int64, _P, c_int64, c_int, c_double, c_double, c_double, _P, c_int64, _P,
                           c_int64, _P, c_int, _P, c_int64, c_int64, _P], 1),
    "gtb_laplacian_count": ([_P, _P, _P, c_int64, _P, _P, _P], 1),
    "gtb_laplacian_fill": ([_P, _P, _P, c_int64, _P, _P, c_int, _P, _P, _P], 1),
    "gtb_row_scale": ([_P, _P, c_int64, c_int, c_int, _P, _P], 1),
    "gtb_slice_f64": ([_P, c_int64, c_int64, c_int64, c_int, c_int, c_int64, c_int64, _P, _P, _P], 2),
    "gtb_gemm_i8": ([_P, _P, c_int, c_int64, c_int64, c_int64, c_int64, c_int64, _P, _P, _P, c_int64, c_int, _P], 1),
    "gtb_dense_to_csr_count": ([_P, c_int64, c_int64, _P, _P], 1),
    "gtb_dense_to_csr_fill": ([_P, c_int64, c_int64, _P, _P, _P, _P], 1),
    "gtb_sp_lengths": ([_P, _P, _P, c_int64, _P, c_int, c_int, c_int, _P, _P, _P], 1),
    "gtb_sp_components": ([_P, _P, c_int64, _P, _P], 3),
    "gtb_sp_traverse": ([_P, _P, _P, c_int64, _P, c_int, c_int, _P, _P, _P], 1),
    "gtb_sp_store_rows": ([_P, c_int, c_int64, _P, c_int, _P, c_int64, _P], 1),
    "gtb_sp_finish": ([_P, c_int64, _P], 1),
}
# entry points whose last pointer arguments are optional: a call may omit them (NULL)
_OPTIONAL_TAIL = {"gtb_knn_topk_tc_seeded": 3}
_PLAIN = {
    "gtb_last_error": ([], ctypes.c_char_p),
    "gtb_version": ([], c_int),
    "gtb_col_mean_ws_doubles": ([c_int], c_int64),
    "gtb_scan_ws_elems": ([c_int64], c_int64),
    "gtb_sym_merge_reg_rows": ([], c_int),
    "gtb_cluster_aggregate_ws_elems": ([c_int], c_int64),
    "gtb_tc_max_kp": ([], c_int),
    "gtb_tc_fp16_maxnorm": ([], c_float),
    "gtb_tc_scratch_bytes": ([c_int64], c_int64),
    "gtb_gemm_max_k": ([], c_int),
    "gtb_knn_seed_k": ([], c_int),
    "gtb_order_ws_elems": ([c_int64, c_int], c_int64),
    "gtb_sp_ws_bytes": ([c_int64, c_int], c_int64),
}


class EngineError(RuntimeError):
    pass


def header_symbols():
    """Every function name declared in include/gtb200.h."""
    with open(HEADER_PATH) as f:
        text = f.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(gtb_[a-z0-9_]+)\s*\(", text)))


def lib():
    """Loads libgtb200.so (built in-tree by __graft_entry__.build / csrc/build.sh)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise EngineError(
                "libgtb200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` "
                "or graphtools_b200/csrc/build.sh -- there is no CPU fallback." % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (argtypes, _) in _SIGS.items():
            fn = getattr(L, name)
            fn.argtypes = argtypes
            fn.restype = c_int
        for name, (argtypes, restype) in _PLAIN.items():
            fn = getattr(L, name)
            fn.argtypes = argtypes
            fn.restype = restype
        _lib = L
    return _lib


def _ptr(x):
    if x is None:
        return None
    if isinstance(x, int):
        return x
    return x.data_ptr()


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream


timing = None  # set to a dict to collect per-entry-point CUDA-event timings (bench.py / profiling)
timing_only = None  # optional set of timing keys: only these entry points are bracketed with events


def timings_ms():
    """Sum of CUDA-event durations per entry point since `timing` was set (synchronises)."""
    import torch
    torch.cuda.synchronize()
    out = {}
    for name, evs in (timing or {}).items():
        out[name] = (len(evs), sum(a.elapsed_time(b) for a, b in evs))
    return out


def call(name, *args):
    """Invoke a compute entry point on the current torch stream; tensors are passed as pointers."""
    global launch_count, kernel_launches
    L = lib()
    key, name = name, name.split("#")[0]         # "entry#tag": same entry point, timed under its own key
    argtypes, nk = _SIGS[name]
    conv = []
    for a, t in zip(args, argtypes):
        conv.append(_ptr(a) if t is _P else a)
    if 0 < len(argtypes) - 1 - len(conv) <= _OPTIONAL_TAIL.get(name, 0):
        conv += [None] * (len(argtypes) - 1 - len(conv))
    assert len(conv) == len(argtypes) - 1, (name, len(conv), len(argtypes))
    timed = timing is not None and (timing_only is None or key in timing_only)
    if timed:
        import torch
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
    rc = getattr(L, name)(*conv, stream_ptr())
    if timed:
        ev1.record()
        timing.setdefault(key, []).append((ev0, ev1))
    if rc != 0:
        raise EngineError("%s failed (%d): %s" % (name, rc, L.gtb_last_error().decode()))
    launch_count += 1
    kernel_launches += nk


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise EngineError("graphtools_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    lib()
