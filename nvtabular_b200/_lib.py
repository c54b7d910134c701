"""ctypes binding of libnvtb200.so (the C-ABI declared in include/nvtb200.h).

This is the only place Python touches native code.  There is NO CPU fallback:
if the shared library is missing, or a call fails, an exception is raised
(``NvtbError``).  Device memory, streams and collectives come from torch; the
kernels come from the library.
"""
import ctypes
import os
import threading
from ctypes import (POINTER, Structure, c_char_p, c_double, c_int, c_int32,
                    c_int64, c_uint8, c_uint64, c_void_p)

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libnvtb200.so")

# nvtb_dtype_t
I32, I64, F32, F64, U8, H64 = 0, 1, 2, 3, 4, 5


class NvtbError(RuntimeError):
    """A libnvtb200 call returned a negative status."""


class nvtb_col_t(Structure):
    _fields_ = [("data", c_void_p), ("validity", c_void_p), ("dtype", c_int32), ("_pad", c_int32)]


class nvtb_vocab_info_t(Structure):
    _fields_ = [("n_kept", c_int64), ("n_total", c_int64), ("null_size", c_int64),
                ("oov_size", c_int64), ("unique_size", c_int64)]


# every exported symbol of include/nvtb200.h with its signature
_SIGNATURES = {
    "nvtb_version": (c_int, []),
    "nvtb_last_error": (c_char_p, []),
    "nvtb_device_sm_count": (c_int, [POINTER(c_int)]),
    "nvtb_moments_init": (c_int, [c_void_p, c_int, c_void_p]),
    "nvtb_moments_accumulate": (c_int, [POINTER(nvtb_col_t), c_int, c_int64, POINTER(c_double), c_void_p, c_void_p]),
    "nvtb_moments_finalize": (c_int, [POINTER(c_double), c_int, POINTER(c_double)]),
    "nvtb_fill_apply": (c_int, [POINTER(nvtb_col_t), c_int, c_int64, POINTER(c_double), POINTER(c_void_p), POINTER(c_void_p), c_void_p]),
    "nvtb_normalize_apply": (c_int, [POINTER(nvtb_col_t), c_int, c_int64, POINTER(c_double), POINTER(c_double), POINTER(c_double), POINTER(c_void_p), c_int, c_void_p]),
    "nvtb_minmax_apply": (c_int, [POINTER(nvtb_col_t), c_int, c_int64, POINTER(c_double), POINTER(c_double), POINTER(c_double), POINTER(c_void_p), c_int, c_void_p]),
    "nvtb_cliplog_apply": (c_int, [POINTER(nvtb_col_t), c_int, c_int64, POINTER(c_double), POINTER(c_double), POINTER(c_double), c_int, POINTER(c_void_p), c_int, c_void_p]),
    "nvtb_hash_bucket_apply": (c_int, [POINTER(nvtb_col_t), c_int, c_int64, c_uint64, c_int64, c_void_p, c_int, c_void_p]),
    "nvtb_hash_values": (c_int, [POINTER(nvtb_col_t), c_int64, c_void_p, c_void_p]),
    "nvtb_hashagg_create": (c_int, [POINTER(c_void_p), c_int, c_int64]),
    "nvtb_hashagg_destroy": (c_int, [c_void_p]),
    "nvtb_hashagg_reset": (c_int, [c_void_p, c_void_p]),
    "nvtb_hashagg_insert": (c_int, [c_void_p, POINTER(nvtb_col_t), POINTER(nvtb_col_t), c_int64, c_void_p]),
    "nvtb_hashagg_merge": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "nvtb_hashagg_add_null_group": (c_int, [c_void_p, c_int64, POINTER(c_double)]),
    "nvtb_hashagg_size": (c_int, [c_void_p, POINTER(c_int64), POINTER(c_int64), c_void_p]),
    "nvtb_hashagg_export": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, POINTER(c_double), c_void_p]),
    "nvtb_hashagg_flush": (c_int, [c_void_p, c_void_p]),
    "nvtb_hashagg_mode": (c_int, [c_void_p, POINTER(c_int)]),
    "nvtb_hashagg_to_sorted": (c_int, [c_void_p, c_void_p]),
    "nvtb_hashagg_export_packed": (c_int, [c_void_p, c_void_p, POINTER(c_int64), c_void_p]),
    "nvtb_pairs_lower_bounds": (c_int, [c_void_p, c_int64, c_void_p, c_int, c_void_p, c_void_p]),
    "nvtb_pairs_merge": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, POINTER(c_int64), c_void_p]),
    "nvtb_segment_copy_u64": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int64, c_void_p]),
    "nvtb_radix_sort_u32": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_int, POINTER(c_int), c_void_p]),
    "nvtb_radix_sort_u64": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_int, POINTER(c_int), c_void_p]),
    "nvtb_partition_by_owner": (c_int, [c_void_p, c_int64, c_int, c_void_p, POINTER(c_int64), c_void_p]),
    "nvtb_partition_by_owner_async": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p]),
    "nvtb_gather_i64": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "nvtb_gather_f64_rows": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "nvtb_pack_keys2": (c_int, [POINTER(nvtb_col_t), POINTER(nvtb_col_t), c_int64, c_void_p, c_void_p, c_void_p]),
    "nvtb_vocab_build": (c_int, [POINTER(c_void_p), c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int64, c_int, c_int64, c_void_p]),
    "nvtb_vocab_build_from_hashagg": (c_int, [POINTER(c_void_p), c_void_p, c_int64, c_int64, c_int64, c_int, c_int64, c_void_p]),
    "nvtb_vocab_build_from_pairs": (c_int, [POINTER(c_void_p), c_void_p, c_int64, c_int64, c_int64, c_int64, c_int64, c_void_p]),
    "nvtb_vocab_from_arrays": (c_int, [POINTER(c_void_p), c_void_p, c_void_p, c_int64, c_void_p]),
    "nvtb_vocab_destroy": (c_int, [c_void_p]),
    "nvtb_vocab_info": (c_int, [c_void_p, POINTER(nvtb_vocab_info_t)]),
    "nvtb_vocab_export": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "nvtb_encode_apply": (c_int, [c_void_p, POINTER(nvtb_col_t), c_int64, c_int64, c_int64, c_int64, c_uint64, POINTER(nvtb_col_t), c_int, c_void_p, c_int, c_void_p]),
    "nvtb_comm_available": (c_int, []),
    "nvtb_comm_unique_id": (c_int, [c_void_p]),
    "nvtb_comm_create": (c_int, [POINTER(c_void_p), c_void_p, c_int, c_int]),
    "nvtb_comm_wrap": (c_int, [POINTER(c_void_p), c_void_p, c_int, c_int]),
    "nvtb_comm_destroy": (c_int, [c_void_p]),
    "nvtb_comm_rank": (c_int, [c_void_p, POINTER(c_int), POINTER(c_int)]),
    "nvtb_comm_allreduce_f64": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    "nvtb_comm_allreduce_i64": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    "nvtb_moments_allreduce": (c_int, [c_void_p, c_void_p, c_int, c_void_p]),
    "nvtb_comm_allgather": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "nvtb_comm_alltoallv": (c_int, [c_void_p, c_void_p, POINTER(c_int64), c_void_p, POINTER(c_int64), c_int, c_void_p]),
    "nvtb_infer_vocab_create": (c_int, [POINTER(c_void_p), c_void_p, c_int64]),
    "nvtb_infer_vocab_from_device": (c_int, [POINTER(c_void_p), c_void_p, c_void_p]),
    "nvtb_infer_vocab_destroy": (c_int, [c_void_p]),
    "nvtb_infer_categorify_host": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int64, c_int64, c_int64, c_int64, c_uint64, c_void_p, c_int, c_int]),
    "nvtb_infer_fill_host": (c_int, [c_void_p, c_int, c_int64, c_double]),
    "nvtb_groupstats_create": (c_int, [POINTER(c_void_p), c_void_p, c_int64, c_void_p, c_int, c_int64, c_void_p]),
    "nvtb_groupstats_destroy": (c_int, [c_void_p]),
    "nvtb_groupstats_gather": (c_int, [c_void_p, POINTER(nvtb_col_t), c_int64, POINTER(c_int), c_int, POINTER(c_double), POINTER(c_void_p), POINTER(c_int), c_void_p]),
    "nvtb_sort_rows": (c_int, [POINTER(nvtb_col_t), POINTER(c_int), c_int, c_int, c_int64, c_void_p, c_void_p, c_void_p]),
    "nvtb_segments": (c_int, [POINTER(nvtb_col_t), c_int, c_void_p, c_int64, c_void_p, c_void_p, POINTER(c_int64), POINTER(c_int64), c_void_p]),
    "nvtb_gather_rows": (c_int, [POINTER(nvtb_col_t), c_void_p, c_void_p, c_int, c_int64, c_void_p, c_void_p, c_void_p]),
    "nvtb_segment_agg": (c_int, [POINTER(nvtb_col_t), c_void_p, c_void_p, c_int64, POINTER(c_void_p), POINTER(c_void_p), c_void_p]),
    "nvtb_segment_sorted_agg": (c_int, [POINTER(nvtb_col_t), c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "nvtb_list_slice_offsets": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int64, c_int64, c_int, c_int64, c_void_p, POINTER(c_int64), c_void_p]),
    "nvtb_list_slice": (c_int, [c_void_p, POINTER(nvtb_col_t), c_int64, c_void_p, c_void_p, c_int, c_int64, c_int64, c_int, c_int64, c_double, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None
_lock = threading.Lock()


def load():
    """Load libnvtb200.so (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise NvtbError(
                f"{LIB_PATH} is missing: build it with `python -m nvtabular_b200._build` "
                "(nvcc, sm_100a). nvtabular_b200 has no CPU fallback.")
        import torch  # noqa: F401  (loads libcudart.so.12 into the process first)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the .so lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc):
    if rc != 0:
        msg = load().nvtb_last_error()
        raise NvtbError(f"libnvtb200 status {rc}: {msg.decode() if msg else '?'}")


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise NvtbError("nvtabular_b200 needs a CUDA device (B200, sm_100a); there is no CPU path")


def stream_ptr():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def col_array(cols):
    """cols: iterable of (data_ptr, validity_ptr_or_None, dtype_code)."""
    cols = list(cols)
    arr = (nvtb_col_t * max(len(cols), 1))()
    for i, (d, v, dt) in enumerate(cols):
        arr[i].data = d
        arr[i].validity = v
        arr[i].dtype = dt
    return arr


def double_array(vals):
    vals = list(vals)
    arr = (c_double * max(len(vals), 1))()
    for i, v in enumerate(vals):
        arr[i] = v
    return arr


def ptr_array(ptrs):
    ptrs = list(ptrs)
    arr = (c_void_p * max(len(ptrs), 1))()
    for i, p in enumerate(ptrs):
        arr[i] = p
    return arr


def int_array(vals):
    vals = list(vals)
    arr = (c_int * max(len(vals), 1))()
    for i, v in enumerate(vals):
        arr[i] = v
    return arr
