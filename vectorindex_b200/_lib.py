"""ctypes binding of ``libvindex_b200.so`` -- the C-ABI CUDA library (include/vindex_cuda.h,
include/cpq_encode.h).  There is no CPU fallback: if the shared library is missing this module raises,
and every entry point fails with ``VIX_ERR_NO_DEVICE`` when no sm_100 GPU is usable.

Buffers may be numpy arrays (host pointers) or torch tensors (host or CUDA device pointers); the library
detects host vs device per pointer.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VIX_LIB_PATH") or os.path.join(_HERE, "libvindex_b200.so")   # override: kernel A/B experiments

VIX_OK = 0
METRIC_L2, METRIC_IP = 0, 1
ORDER_MIN, ORDER_MAX = 0, 1
INDEX_FLAT, INDEX_IVF_FLAT, INDEX_IVF_PQ = 0, 1, 2
MAX_K = 512
MAX_K_LARGE = 16384          # k-NN search beyond MAX_K: the exact two-pass route over the range-search scans

STATUS_NAMES = {
    0: "ok", -1: "invalidDim", -2: "invalidK", -3: "nullPtr", -4: "invalidLayout", -5: "invalidParameter",
    -6: "notTrained", -7: "emptyInput", -8: "contractViolation", -9: "unsupported", -100: "cudaError",
    -101: "noDevice", -102: "outOfMemory", 1: "noConvergence",
}


class VectorIndexError(RuntimeError):
    """Mirror of the reference's ``VectorIndexError(kind:message:)`` (ErrorHandling/VectorIndexError.swift)."""

    def __init__(self, status: int, message: str):
        self.status = status
        self.kind = STATUS_NAMES.get(status, str(status))
        super().__init__(f"[{self.kind}] {message}")


class PQEncodeOpts(C.Structure):
    """cpq_encode.h PQEncodeOpts (reference: Sources/CPQEncode/include/cpq_encode.h:30-38)."""
    _fields_ = [("layout", C.c_int), ("use_dot_trick", C.c_bool), ("precompute_x_norm2", C.c_bool),
                ("prefetch_distance", C.c_int), ("num_threads", C.c_int), ("soa_block_B", C.c_int),
                ("interleave_g", C.c_int)]


class PQLutOpts(C.Structure):
    _fields_ = [("use_dot_trick", C.c_int), ("include_q_norm", C.c_bool), ("strict_fp", C.c_bool)]


class ADCScanOpts(C.Structure):
    _fields_ = [("layout", C.c_int), ("group_size", C.c_int), ("stride", C.c_int), ("add_bias", C.c_float),
                ("strict_fp", C.c_bool)]


class KMeansCfg(C.Structure):
    _fields_ = [("batch_size", C.c_int), ("epochs", C.c_int), ("tol", C.c_float), ("seed", C.c_uint64),
                ("stream_id", C.c_uint64), ("compute_assignments", C.c_bool), ("mode", C.c_int)]


class PQTrainCfg(C.Structure):
    _fields_ = [("algorithm", C.c_int), ("max_iters", C.c_int), ("tol", C.c_float), ("batch_size", C.c_int),
                ("sample_n", C.c_int64), ("seed", C.c_uint64), ("stream_id", C.c_int), ("empty_policy", C.c_int),
                ("mode", C.c_int)]


class IndexParams(C.Structure):
    _fields_ = [("kind", C.c_int), ("d", C.c_int), ("metric", C.c_int), ("nlist", C.c_int), ("nprobe", C.c_int),
                ("m", C.c_int), ("ks", C.c_int), ("shard_rank", C.c_int), ("shard_world", C.c_int)]


class SearchStats(C.Structure):
    _fields_ = [("codes_scanned", C.c_int64), ("code_bytes_scanned", C.c_int64), ("ms_coarse", C.c_float),
                ("ms_scan", C.c_float), ("ms_total", C.c_float), ("cycles_prologue", C.c_int64), ("cycles_scan", C.c_int64),
                ("cycles_tail", C.c_int64), ("cycles_select", C.c_int64), ("cycles_probe_table", C.c_int64),
                ("cycles_lut", C.c_int64), ("merge_candidates", C.c_int64), ("ms_scan_kernel", C.c_float), ("scan_path", C.c_int32)]


_LIB = None

# symbol -> (restype, is_status)
_EXPORTS = [
    "vix_version", "vix_last_error", "vix_clear_error", "vix_device_count", "vix_set_device", "vix_set_stream", "vix_set_async", "vix_get_async",
    "vix_synchronize", "vix_kernel_launches", "vix_scan_tc_launches", "vix_tc_shortlist_calls", "vix_tc_shortlist_exact_rows",
    "vix_l2sqr_f32_block", "vix_ip_f32_block", "vix_row_norms_f32", "vix_flat_search_f32", "vix_select_topk_f32",
    "vix_merge_topk_f32", "vix_rerank_exact_topk_f32", "vix_centroid_batch_score_f32", "vix_ivf_select_nprobe_batch_f32", "vix_ivf_assign_f32",
    "vix_ivf_assign_metric_f32", "vix_pq_query_subnorms_f32", "vix_pq_lut_batch_l2_f32", "vix_pq_lut_residual_l2_f32", "vix_adc_scan_u8",
    "vix_adc_scan_u4", "vix_kmeanspp_seed_f32", "vix_kmeans_minibatch_f32", "vix_pq_train_f32", "vix_pq_train_streaming_f32",
    "vix_index_params_default", "vix_index_create", "vix_index_destroy", "vix_index_train", "vix_index_set_coarse",
    "vix_index_set_codebooks", "vix_index_get_coarse", "vix_index_get_codebooks", "vix_index_add", "vix_index_remove",
    "vix_index_import_lists", "vix_index_count", "vix_index_list_sizes", "vix_index_export_lists", "vix_index_clear",
    "vix_index_search", "vix_index_search_ex", "vix_index_search_rerank", "vix_index_trace", "vix_index_trace_get", "vix_index_probe_range", "vix_index_search_with_probes",
    "vix_index_search_with_probes_ex", "vix_index_search_filtered", "vix_index_range_search", "vix_range_result_nq",
    "vix_range_result_total", "vix_range_result_get", "vix_range_result_destroy",
    "vix_comm_unique_id", "vix_comm_create", "vix_comm_destroy", "vix_comm_rank", "vix_comm_world",
    "vix_comm_uses_peer_memory", "vix_comm_trace", "vix_comm_trace_get", "vix_sharded_query_block", "vix_sharded_add", "vix_sharded_search",
    "vix_sharded_search_filtered", "vix_sharded_range_search", "vix_debug_shard_range_merge", "vix_debug_shard_knn_merge",
    "vix_debug_shard_flat_merge", "vix_debug_sharded_emulate", "vix_replicated_add", "vix_replicated_search",
    "vix_replicated_search_filtered", "vix_replicated_range_search", "vix_debug_replica_assemble",
    "vix_index_encode", "vix_index_add_encoded", "vix_debug_tc_scores_f32", "vix_debug_tc_codes", "vix_debug_tc_seed", "vix_debug_shard_merge", "vix_accel_rank_candidates_f32",
    "cpq_encode_u8_f32", "cpq_encode_u8_f32_with_csq", "cpq_encode_u4_f32", "cpq_encode_residual_u8_f32",
    "cpq_encode_residual_u8_f32_with_csq", "cpq_encode_residual_u4_f32", "cpq_pack_u4_bulk", "cpq_unpack_u4_bulk",
]


def exported_symbols():
    """Every symbol include/*.h declares (tests check that the library exports all of them)."""
    return list(_EXPORTS)


def lib() -> C.CDLL:
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `make -C vectorindex_b200/csrc` "
                "(or `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        L.vix_last_error.restype = C.c_char_p
        L.vix_kernel_launches.restype = C.c_int64
        L.vix_scan_tc_launches.restype = C.c_int64
        L.vix_tc_shortlist_calls.restype = C.c_int64
        L.vix_tc_shortlist_exact_rows.restype = C.c_int64
        L.vix_index_count.restype = C.c_int64
        L.vix_range_result_nq.restype = C.c_int64
        L.vix_range_result_total.restype = C.c_int64
        L.vix_range_result_destroy.restype = None
        L.vix_index_destroy.restype = None
        L.vix_index_params_default.restype = None
        L.vix_clear_error.restype = None
        for name in _EXPORTS:
            if name.startswith("cpq_"):
                getattr(L, name).restype = None
        _LIB = L
    return _LIB


def last_error() -> str:
    return (lib().vix_last_error() or b"").decode("utf-8", "replace")


def check(status: int, allow=(0,)):
    if status not in allow:
        raise VectorIndexError(status, last_error())
    return status


def clear_error():
    lib().vix_clear_error()


# ------------------------------------------------------------------------------------------------
# pointer marshalling
# ------------------------------------------------------------------------------------------------
def _is_torch(a) -> bool:
    return type(a).__module__.startswith("torch")


def ptr(a, dtype=None):
    """void* of a numpy array / torch tensor (must be contiguous), or NULL for None."""
    if a is None:
        return C.c_void_p(0)
    if _is_torch(a):
        if not a.is_contiguous():
            raise ValueError("tensor must be contiguous")
        if dtype is not None:
            import torch
            want = {np.float32: torch.float32, np.int32: torch.int32, np.int64: torch.int64, np.uint8: torch.uint8,
                    np.uint64: torch.int64}[dtype]
            if a.dtype != want:
                raise TypeError(f"tensor dtype {a.dtype} != {want}")
        return C.c_void_p(a.data_ptr())
    if not isinstance(a, np.ndarray):
        raise TypeError(f"expected numpy array or torch tensor, got {type(a)}")
    if not a.flags["C_CONTIGUOUS"]:
        raise ValueError("array must be C-contiguous")
    if dtype is not None and a.dtype != np.dtype(dtype):
        raise TypeError(f"array dtype {a.dtype} != {np.dtype(dtype)}")
    return C.c_void_p(a.ctypes.data)


def as_input(a, dtype):
    """Contiguous array / tensor of ``dtype`` (converted when it is not; stays on its device)."""
    if a is None:
        return None
    if _is_torch(a):
        import torch
        want = {np.float32: torch.float32, np.int32: torch.int32, np.int64: torch.int64, np.uint8: torch.uint8,
                np.uint64: torch.int64}.get(dtype)
        if want is not None and a.dtype != want:       # e.g. int32 ids: the C side reads int64
            a = a.to(want)
        return a.contiguous()
    return np.ascontiguousarray(a, dtype=dtype)


def empty_like_input(ref, shape, dtype):
    """Output buffer living where ``ref`` lives (torch CUDA tensor -> CUDA tensor, else numpy)."""
    if _is_torch(ref):
        import torch
        tdt = {np.float32: torch.float32, np.int32: torch.int32, np.int64: torch.int64, np.uint8: torch.uint8,
               np.uint64: torch.int64}[dtype]              # torch carries the 64 key bits in int64 tensors
        return torch.empty(shape, dtype=tdt, device=ref.device)
    return np.empty(shape, dtype=dtype)
