"""Thin, typed Python face of the C-ABI (include/nvtb200.h): every function
here is one or two calls into libnvtb200.so on Column buffers.  The operator
classes in nvtabular_b200/ops are written against this module only.

No arithmetic happens in Python on row data; torch is used to allocate output
buffers and to read back O(#columns) scalars.
"""
import ctypes
from ctypes import byref, c_int, c_int64, c_void_p
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _lib
from .column import Column

_CODE2TORCH = {_lib.I32: torch.int32, _lib.I64: torch.int64, _lib.F32: torch.float32,
               _lib.F64: torch.float64, _lib.U8: torch.uint8}
_NP2CODE = {np.dtype("int32"): _lib.I32, np.dtype("int64"): _lib.I64,
            np.dtype("float32"): _lib.F32, np.dtype("float64"): _lib.F64,
            np.dtype("uint8"): _lib.U8, np.dtype("bool"): _lib.U8}
NAN = float("nan")
kernel_launches = 0  # counted for bench.py's "gpu_launches"


def _count(n=1):
    global kernel_launches
    kernel_launches += n


# --- optional per-kernel-family device timing (bench.py's roofline object) -----
# When `profile` is a list, every wrapper below brackets its launch with CUDA
# events on the launching stream and appends (family, start, end, algorithmic
# bytes).  Events are only read after the timed region has been synchronised.
profile = None


class _timed:
    def __init__(self, family: str, nbytes: float):
        self.family, self.nbytes = family, nbytes

    def __enter__(self):
        if profile is not None:
            self.s = torch.cuda.Event(enable_timing=True)
            self.e = torch.cuda.Event(enable_timing=True)
            self.s.record()
        return self

    def __exit__(self, *exc):
        if profile is not None:
            self.e.record()
            profile.append((self.family, self.s, self.e, self.nbytes))
        return False


def _in_bytes(cols) -> float:
    """algorithmic read bytes: data + 1 validity bit per row (SURVEY.md §8d)."""
    return float(sum(c.data.numel() * (c.data.element_size() + 0.125) for c in cols))


def dtype_code(dt) -> int:
    if isinstance(dt, torch.dtype):
        return {v: k for k, v in _CODE2TORCH.items()}[dt]
    return _NP2CODE[np.dtype(dt)]


def _ptr(t: Optional[torch.Tensor]):
    return c_void_p(t.data_ptr()) if t is not None and t.numel() else None


def _fills(cols: Sequence[Column]):
    return _lib.double_array([NAN if c.fill is None else float(c.fill) for c in cols])


def _descs(cols: Sequence[Column]):
    return _lib.col_array([c.desc() for c in cols])


def _check_same_len(cols: Sequence[Column]) -> int:
    n = cols[0].data.numel()
    for c in cols:
        if c.data.numel() != n:
            raise ValueError("columns of one call must have the same length")
    return n


# ----------------------------------------------------------------- moments
class Moments:
    """Running {count, sum, sumsq, min, max} per column on the device
    (nvtb_moments_*; replaces nvtabular/ops/moments.py:28-116)."""

    def __init__(self, ncols: int, device=None):
        _lib.require_cuda()
        self.lib = _lib.load()
        self.ncols = ncols
        self.acc = torch.empty(ncols * 5, dtype=torch.float64, device=device or "cuda")
        _lib.check(self.lib.nvtb_moments_init(_ptr(self.acc), ncols, _lib.stream_ptr()))
        _count()

    def accumulate(self, cols: Sequence[Column]):
        assert len(cols) == self.ncols
        n = _check_same_len(cols)
        with _timed("moments", _in_bytes(cols)):
            _lib.check(self.lib.nvtb_moments_accumulate(
                _descs(cols), self.ncols, n, _fills(cols), _ptr(self.acc), _lib.stream_ptr()))
        _count(2)

    def allreduce(self):
        """Cross-GPU merge: one NCCL all-reduce of 3 sums + min + max per column
        (SURVEY.md §8e; replaces the dask tree of moments.py:45-55)."""
        import torch.distributed as dist
        from .dist import native_comm, world
        if world()[0] <= 1:
            return
        nc = native_comm()
        if nc is not None and self.acc.is_cuda:            # the library's own communicator (csrc/comm.cu)
            _lib.check(nc[0].nvtb_moments_allreduce(nc[1], _ptr(self.acc), self.ncols, _lib.stream_ptr()))
            _count()
            return
        a = self.acc.view(self.ncols, 5)
        sums = a[:, 0:3].contiguous()
        mn = a[:, 3].contiguous()
        mx = a[:, 4].contiguous()
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
        dist.all_reduce(mn, op=dist.ReduceOp.MIN)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        a[:, 0:3] = sums
        a[:, 3] = mn
        a[:, 4] = mx

    def result(self):
        """-> dict of numpy arrays: count,sum,sumsq,min,max,mean,var,std."""
        acc = self.acc.cpu().numpy().astype(np.float64)
        out = np.zeros(self.ncols * 3, dtype=np.float64)
        _lib.check(self.lib.nvtb_moments_finalize(
            acc.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), self.ncols,
            out.ctypes.data_as(ctypes.POINTER(ctypes.c_double))))
        a = acc.reshape(self.ncols, 5)
        o = out.reshape(self.ncols, 3)
        return {"count": a[:, 0], "sum": a[:, 1], "sumsq": a[:, 2], "min": a[:, 3], "max": a[:, 4],
                "mean": o[:, 0], "var": o[:, 1], "std": o[:, 2]}


# ------------------------------------------------------------- transforms
def _alloc_like(cols: Sequence[Column], dtype: torch.dtype) -> List[torch.Tensor]:
    return [torch.empty(c.data.numel(), dtype=dtype, device=c.data.device) for c in cols]


def fill_apply(cols: Sequence[Column], fill_vals: Sequence[float], add_binary_cols=False):
    """FillMissing (nvtb_fill_apply).  Returns (filled columns, indicator columns|None)."""
    _lib.require_cuda()
    lib = _lib.load()
    n = _check_same_len(cols)
    outs = [torch.empty_like(c.data) for c in cols]
    flags = [torch.empty(n, dtype=torch.uint8, device=c.data.device) for c in cols] if add_binary_cols else None
    _lib.check(lib.nvtb_fill_apply(
        _descs(cols), len(cols), n, _lib.double_array(fill_vals),
        _lib.ptr_array([o.data_ptr() for o in outs]),
        _lib.ptr_array([f.data_ptr() for f in flags]) if flags else None, _lib.stream_ptr()))
    _count()
    out_cols = [Column(o, None, c.offsets, None, None, c.is_bool) for o, c in zip(outs, cols)]
    flag_cols = [Column(f, None, c.offsets, is_bool=True) for f, c in zip(flags, cols)] if flags else None
    return out_cols, flag_cols


def normalize_apply(cols: Sequence[Column], means, stds, out_dtype=np.float64):
    _lib.require_cuda()
    lib = _lib.load()
    n = _check_same_len(cols)
    code = dtype_code(out_dtype)
    outs = _alloc_like(cols, _CODE2TORCH[code])
    with _timed("normalize", _in_bytes(cols) + sum(o.numel() * o.element_size() for o in outs)):
        _lib.check(lib.nvtb_normalize_apply(
            _descs(cols), len(cols), n, _fills(cols), _lib.double_array(means), _lib.double_array(stds),
            _lib.ptr_array([o.data_ptr() for o in outs]), code, _lib.stream_ptr()))
    _count()
    return [Column(o, None if c.fill is not None else c.validity, c.offsets) for o, c in zip(outs, cols)]


def minmax_apply(cols: Sequence[Column], mins, maxs, out_dtype=np.float64):
    _lib.require_cuda()
    lib = _lib.load()
    n = _check_same_len(cols)
    code = dtype_code(out_dtype)
    outs = _alloc_like(cols, _CODE2TORCH[code])
    _lib.check(lib.nvtb_minmax_apply(
        _descs(cols), len(cols), n, _fills(cols), _lib.double_array(mins), _lib.double_array(maxs),
        _lib.ptr_array([o.data_ptr() for o in outs]), code, _lib.stream_ptr()))
    _count()
    return [Column(o, None if c.fill is not None else c.validity, c.offsets) for o, c in zip(outs, cols)]


def cliplog_apply(cols: Sequence[Column], min_value=None, max_value=None, take_log=False, out_dtype=np.float32):
    """Clip (+ LogOp) with an upstream FillMissing fused in (nvtb_cliplog_apply).  take_log=False
    keeps every column's dtype; nulls that are not filled stay nulls."""
    _lib.require_cuda()
    lib = _lib.load()
    n = _check_same_len(cols)
    code = dtype_code(out_dtype) if take_log else 0
    outs = _alloc_like(cols, _CODE2TORCH[code]) if take_log else [torch.empty_like(c.data) for c in cols]
    lo = _lib.double_array([NAN if min_value is None else float(min_value)] * len(cols))
    hi = _lib.double_array([NAN if max_value is None else float(max_value)] * len(cols))
    with _timed("cliplog", _in_bytes(cols) + sum(o.numel() * o.element_size() for o in outs)):
        _lib.check(lib.nvtb_cliplog_apply(_descs(cols), len(cols), n, _fills(cols), lo, hi, 1 if take_log else 0,
                                          _lib.ptr_array([o.data_ptr() for o in outs]), code, _lib.stream_ptr()))
    _count()
    return [Column(o, None if c.fill is not None else c.validity, c.offsets, None, None, c.is_bool and not take_log)
            for o, c in zip(outs, cols)]


def hash_bucket(cols: Sequence[Column], num_buckets: int, add: int = 0, out_dtype=np.int32) -> torch.Tensor:
    """hash(cols...) % num_buckets + add (nvtb_hash_bucket_apply)."""
    _lib.require_cuda()
    lib = _lib.load()
    n = _check_same_len(cols)
    code = dtype_code(out_dtype)
    out = torch.empty(n, dtype=_CODE2TORCH[code], device=cols[0].data.device)
    with _timed("hash_bucket", _in_bytes(cols) + out.numel() * out.element_size()):
        _lib.check(lib.nvtb_hash_bucket_apply(_descs(cols), len(cols), n, int(num_buckets), int(add),
                                              _ptr(out), code, _lib.stream_ptr()))
    _count()
    return out


def hash_values(col: Column) -> torch.Tensor:
    """raw uint64 value hashes as an int64 tensor (bit pattern)."""
    _lib.require_cuda()
    lib = _lib.load()
    n = col.data.numel()
    out = torch.empty(n, dtype=torch.int64, device=col.data.device)
    _lib.check(lib.nvtb_hash_values(_descs([col]), n, _ptr(out), _lib.stream_ptr()))
    _count()
    return out


def pack_keys2(a: Column, b: Column) -> Column:
    """(a, b) int32 pair -> one order-preserving int64 key column."""
    _lib.require_cuda()
    lib = _lib.load()
    n = _check_same_len([a, b])
    keys = torch.empty(n, dtype=torch.int64, device=a.data.device)
    need_mask = a.validity is not None and b.validity is not None
    nbytes = (((n + 7) // 8 + 31) // 32) * 32
    mask = torch.zeros(nbytes, dtype=torch.uint8, device=a.data.device) if need_mask else None
    _lib.check(lib.nvtb_pack_keys2(_descs([a]), _descs([b]), n, _ptr(keys), _ptr(mask), _lib.stream_ptr()))
    _count()
    return Column(keys, mask)


def unpack_keys2(keys: np.ndarray):
    """host inverse of pack_keys2: int64 -> (a int32, b int32); INT32_MIN marks a null component."""
    k = keys.astype(np.int64)
    a = (k >> 32).astype(np.int32)
    b = ((k & 0xFFFFFFFF).astype(np.uint32) ^ np.uint32(0x80000000)).astype(np.uint32).view(np.int32)
    return a, b


# ------------------------------------------------------------- hash aggregation
class HashAgg:
    """groupby(key, dropna=False) -> size [, sum/sumsq/min/max per cont col]
    (nvtb_hashagg_*; replaces nvtabular/ops/categorify.py:955-1137)."""

    def __init__(self, n_agg: int = 0, capacity_hint: int = 0):
        _lib.require_cuda()
        self.lib = _lib.load()
        self.n_agg = n_agg
        self.h = c_void_p()
        _lib.check(self.lib.nvtb_hashagg_create(byref(self.h), n_agg, int(capacity_hint)))

    def __del__(self):
        try:
            if getattr(self, "h", None) is not None and self.h.value:
                self.lib.nvtb_hashagg_destroy(self.h)
                self.h = c_void_p()
        except Exception:
            pass

    def reset(self):
        _lib.check(self.lib.nvtb_hashagg_reset(self.h, _lib.stream_ptr()))
        _count(2)

    @property
    def mode(self) -> int:
        """0 = resident hash table, 1 = sorted accumulator (csrc/sortagg.cuh)"""
        m = c_int(0)
        _lib.check(self.lib.nvtb_hashagg_mode(self.h, byref(m)))
        return m.value

    def flush(self):
        """fold in whatever a sorted accumulator has staged (timed with the inserts: it is their cost)"""
        with _timed("hashagg_insert", 0.0):
            _lib.check(self.lib.nvtb_hashagg_flush(self.h, _lib.stream_ptr()))
        _count(12)

    def to_sorted(self):
        """make the handle a sorted accumulator (key-ordered packed pairs), see csrc/sortagg.cuh"""
        _lib.check(self.lib.nvtb_hashagg_to_sorted(self.h, _lib.stream_ptr()))
        _count(3)

    def export_packed(self, device="cuda") -> torch.Tensor:
        """packed pairs (key ^ 2^31) << 32 | count of a sorted accumulator, key order, as the bit
        pattern of an int64 tensor"""
        n = c_int64(0)
        _lib.check(self.lib.nvtb_hashagg_export_packed(self.h, None, byref(n), _lib.stream_ptr()))
        out = torch.empty(n.value, dtype=torch.int64, device=device)
        if n.value:
            _lib.check(self.lib.nvtb_hashagg_export_packed(self.h, _ptr(out), byref(n), _lib.stream_ptr()))
        return out

    def insert(self, key: Column, agg_cols: Sequence[Column] = ()):
        n = key.data.numel()
        assert len(agg_cols) == self.n_agg
        for c in agg_cols:
            assert c.data.numel() == n
        with _timed("hashagg_insert", _in_bytes([key]) + _in_bytes(agg_cols)):
            _lib.check(self.lib.nvtb_hashagg_insert(
                self.h, _descs([key]), _descs(agg_cols) if self.n_agg else None, n, _lib.stream_ptr()))
        _count(1)

    def merge(self, keys: torch.Tensor, sizes: torch.Tensor, vals: Optional[torch.Tensor] = None):
        n = keys.numel()
        _lib.check(self.lib.nvtb_hashagg_merge(self.h, _ptr(keys), _ptr(sizes), _ptr(vals), n, _lib.stream_ptr()))
        _count(1 if n else 0)

    def add_null_group(self, size: int, vals: Optional[np.ndarray] = None):
        arr = _lib.double_array(list(vals)) if vals is not None and self.n_agg else None
        _lib.check(self.lib.nvtb_hashagg_add_null_group(self.h, int(size), arr))

    def size(self):
        nu, ns = c_int64(0), c_int64(0)
        _lib.check(self.lib.nvtb_hashagg_size(self.h, byref(nu), byref(ns), _lib.stream_ptr()))
        return nu.value, ns.value

    def export(self, device="cuda"):
        """-> (keys int64[U], sizes int64[U], vals float64[U, n_agg, 4] | None,
                null_size, null_vals ndarray[n_agg,4] | None), unordered."""
        nu, ns = self.size()
        keys = torch.empty(nu, dtype=torch.int64, device=device)
        sizes = torch.empty(nu, dtype=torch.int64, device=device)
        vals = torch.empty((nu, self.n_agg, 4), dtype=torch.float64, device=device) if self.n_agg else None
        null_vals = (ctypes.c_double * (4 * max(self.n_agg, 1)))()
        with _timed("hashagg_export", float(nu * 16)):
            _lib.check(self.lib.nvtb_hashagg_export(self.h, _ptr(keys), _ptr(sizes), _ptr(vals),
                                                    null_vals if self.n_agg else None, _lib.stream_ptr()))
        _count()
        nv = np.array(list(null_vals), dtype=np.float64).reshape(-1, 4)[: self.n_agg] if self.n_agg else None
        return keys, sizes, vals, ns, nv


def partition_by_owner(keys: torch.Tensor, n_parts: int):
    """-> (perm int64[n], counts list[int]) grouping rows by hash-owner."""
    lib = _lib.load()
    n = keys.numel()
    perm = torch.empty(n, dtype=torch.int64, device=keys.device)
    counts = (c_int64 * n_parts)()
    _lib.check(lib.nvtb_partition_by_owner(_ptr(keys), n, n_parts, _ptr(perm), counts, _lib.stream_ptr()))
    _count(2)
    return perm, [int(c) for c in counts]


def partition_by_owner_async(keys: torch.Tensor, n_parts: int, counts_out: torch.Tensor):
    """-> perm int64[n]; the per-owner row counts go to `counts_out` (device int64[n_parts])
    without a host round trip."""
    lib = _lib.load()
    n = keys.numel()
    perm = torch.empty(n, dtype=torch.int64, device=keys.device)
    _lib.check(lib.nvtb_partition_by_owner_async(_ptr(keys), n, n_parts, _ptr(perm), _ptr(counts_out),
                                                 _lib.stream_ptr()))
    _count(3)
    return perm


def gather_i64(src: torch.Tensor, perm: torch.Tensor) -> torch.Tensor:
    lib = _lib.load()
    out = torch.empty(perm.numel(), dtype=torch.int64, device=src.device)
    _lib.check(lib.nvtb_gather_i64(_ptr(src), _ptr(perm), perm.numel(), _ptr(out), _lib.stream_ptr()))
    _count()
    return out


def gather_f64_rows(src: torch.Tensor, perm: torch.Tensor, width: int) -> torch.Tensor:
    lib = _lib.load()
    out = torch.empty((perm.numel(), width), dtype=torch.float64, device=src.device)
    _lib.check(lib.nvtb_gather_f64_rows(_ptr(src), _ptr(perm), perm.numel(), width, _ptr(out), _lib.stream_ptr()))
    _count()
    return out


# ------------------------------------------------------------------ vocabulary
class Vocab:
    """Ordered vocabulary + device lookup (nvtb_vocab_*; replaces
    _write_uniques/_save_encodings/_encode, categorify.py:1149-1337,719-822,1558-1807)."""

    def __init__(self, handle, lib, n_total=None):
        self.h = handle
        self.lib = lib
        self._info = None
        self._n_total = n_total

    def _load(self):
        """nvtb_vocab_build only ENQUEUES the build; the scalars come back through a pinned
        mailbox and are read (one event wait) the first time anything asks for them."""
        if self._info is None:
            info = _lib.nvtb_vocab_info_t()
            _lib.check(self.lib.nvtb_vocab_info(self.h, byref(info)))
            self._info = info
        return self._info

    n_kept = property(lambda self: self._load().n_kept)
    null_size = property(lambda self: self._load().null_size)
    oov_size = property(lambda self: self._load().oov_size)
    unique_size = property(lambda self: self._load().unique_size)

    @property
    def n_total(self):
        return self._n_total if self._n_total is not None else self._load().n_total

    @classmethod
    def build(cls, keys: torch.Tensor, sizes: torch.Tensor, null_size=0, freq_threshold=0,
              max_size=0, num_buckets=0, key_bits=0, size_bound=0):
        _lib.require_cuda()
        lib = _lib.load()
        h = c_void_p()
        with _timed("vocab_build", float(keys.numel() * 16)):
            _lib.check(lib.nvtb_vocab_build(byref(h), _ptr(keys), _ptr(sizes), keys.numel(), int(null_size),
                                            int(freq_threshold or 0), int(max_size or 0), int(num_buckets or 0),
                                            int(key_bits), int(size_bound), _lib.stream_ptr()))
        _count(8)
        return cls(h, lib, n_total=keys.numel())

    @classmethod
    def build_from_agg(cls, agg: "HashAgg", freq_threshold=0, max_size=0, num_buckets=0, key_bits=0,
                       size_bound=0):
        """vocabulary straight from a group-by handle (single GPU): no int64 export round
        trip; a sorted accumulator only needs one stable sort on the size bits."""
        _lib.require_cuda()
        lib = _lib.load()
        h = c_void_p()
        with _timed("vocab_build", 0.0):
            _lib.check(lib.nvtb_vocab_build_from_hashagg(byref(h), agg.h, int(freq_threshold or 0), int(max_size or 0),
                                                         int(num_buckets or 0), int(key_bits), int(size_bound),
                                                         _lib.stream_ptr()))
        _count(8)
        return cls(h, lib)

    @classmethod
    def build_from_pairs(cls, ordered_pairs: torch.Tensor, null_size=0, freq_threshold=0, max_size=0, num_buckets=0):
        """vocabulary from packed pairs already in (count desc, key asc) order (cross-GPU merge)"""
        _lib.require_cuda()
        lib = _lib.load()
        h = c_void_p()
        with _timed("vocab_build", float(ordered_pairs.numel() * 16)):
            _lib.check(lib.nvtb_vocab_build_from_pairs(byref(h), _ptr(ordered_pairs), ordered_pairs.numel(),
                                                       int(null_size), int(freq_threshold or 0), int(max_size or 0),
                                                       int(num_buckets or 0), _lib.stream_ptr()))
        _count(4)
        return cls(h, lib, n_total=ordered_pairs.numel())

    @classmethod
    def from_arrays(cls, keys: torch.Tensor, sizes: Optional[torch.Tensor] = None):
        _lib.require_cuda()
        lib = _lib.load()
        h = c_void_p()
        _lib.check(lib.nvtb_vocab_from_arrays(byref(h), _ptr(keys), _ptr(sizes), keys.numel(), _lib.stream_ptr()))
        _count(2)
        return cls(h, lib)

    def __del__(self):
        try:
            if getattr(self, "h", None) is not None and self.h.value:
                self.lib.nvtb_vocab_destroy(self.h)
                self.h = c_void_p()
        except Exception:
            pass

    def export(self, device="cuda", with_sizes=True):
        keys = torch.empty(self.n_kept, dtype=torch.int64, device=device)
        sizes = torch.empty(self.n_kept, dtype=torch.int64, device=device) if with_sizes else None
        _lib.check(self.lib.nvtb_vocab_export(self.h, _ptr(keys), _ptr(sizes), _lib.stream_ptr()))
        return keys, sizes

    def encode(self, key: Column, null_label=1, oov_label=2, first_label=3, num_buckets=0,
               hash_cols: Sequence[Column] = (), out_dtype=np.int64) -> torch.Tensor:
        n = key.data.numel()
        code = dtype_code(out_dtype)
        out = torch.empty(n, dtype=_CODE2TORCH[code], device=key.data.device)
        with _timed("encode", _in_bytes([key]) + out.numel() * out.element_size()):
            _lib.check(self.lib.nvtb_encode_apply(
                self.h, _descs([key]), n, int(null_label), int(oov_label), int(first_label),
                int(num_buckets or 0), _descs(hash_cols) if hash_cols else None, len(hash_cols),
                _ptr(out), code, _lib.stream_ptr()))
        _count()
        return out


def pairs_lower_bounds(pairs: torch.Tensor, bounds: torch.Tensor) -> torch.Tensor:
    """number of key-sorted packed pairs whose unsigned key is below each of `bounds` (int64
    tensor of values in [0, 2^32]; 2^32 = "everything") -> int64 tensor on the device"""
    lib = _lib.load()
    n = pairs.numel()
    full = bounds >= (1 << 32)
    b = torch.where(full, torch.zeros_like(bounds), bounds)
    b32 = torch.where(b >= (1 << 31), b - (1 << 32), b).to(torch.int32).contiguous()
    out = torch.empty(bounds.numel(), dtype=torch.int64, device=pairs.device)
    _lib.check(lib.nvtb_pairs_lower_bounds(_ptr(pairs), n, _ptr(b32), b32.numel(), _ptr(out), _lib.stream_ptr()))
    _count()
    return torch.where(full, torch.full_like(out, n), out)


def pairs_merge(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """merge of two key-sorted, key-unique packed-pair arrays, counts of equal keys added"""
    lib = _lib.load()
    out = torch.empty(a.numel() + b.numel(), dtype=torch.int64, device=a.device)
    n = c_int64(0)
    _lib.check(lib.nvtb_pairs_merge(_ptr(a), a.numel(), _ptr(b), b.numel(), _ptr(out), byref(n), _lib.stream_ptr()))
    _count(4)
    return out[: n.value]


def segment_copy(src: torch.Tensor, dst: torch.Tensor, seg_src: torch.Tensor, seg_dst: torch.Tensor):
    """dst[seg_dst[s] + k] = src[seg_src[s] + k] for every segment s (seg_src: nseg + 1 ascending
    offsets ending at src.numel(); seg_dst < 0 skips a segment)"""
    lib = _lib.load()
    _lib.check(lib.nvtb_segment_copy_u64(_ptr(src), _ptr(dst), _ptr(seg_src), _ptr(seg_dst), seg_dst.numel(),
                                         src.numel(), _lib.stream_ptr()))
    _count()


def radix_sort(data: torch.Tensor, lo_bit: int = 0, hi_bit: Optional[int] = None, descending=False) -> torch.Tensor:
    """stable LSD radix sort of an int32/int64 tensor by bits [lo_bit, hi_bit) of its
    elements viewed as unsigned (nvtb_radix_sort_u32/u64); returns the sorted tensor"""
    _lib.require_cuda()
    lib = _lib.load()
    assert data.dtype in (torch.int32, torch.int64) and data.is_contiguous()
    bits = 8 * data.element_size()
    hi_bit = bits if hi_bit is None else hi_bit
    a = data.clone()
    b = torch.empty_like(a)
    flag = c_int(0)
    fn = lib.nvtb_radix_sort_u32 if bits == 32 else lib.nvtb_radix_sort_u64
    _lib.check(fn(_ptr(a), _ptr(b), a.numel(), int(lo_bit), int(hi_bit), 1 if descending else 0, byref(flag),
                  _lib.stream_ptr()))
    _count(3)
    return b if flag.value else a


class GroupStats:
    """key -> row of a stats matrix, gathered per row (nvtb_groupstats_*)."""

    def __init__(self, keys: torch.Tensor, stats: torch.Tensor, null_row: int = -1):
        _lib.require_cuda()
        self.lib = _lib.load()
        self.h = c_void_p()
        stats = stats.contiguous().to(torch.float64)
        self.width = int(stats.shape[1])
        _lib.check(self.lib.nvtb_groupstats_create(byref(self.h), _ptr(keys), keys.numel(), _ptr(stats),
                                                   self.width, int(null_row), _lib.stream_ptr()))
        _count(2)

    def __del__(self):
        try:
            if getattr(self, "h", None) is not None and self.h.value:
                self.lib.nvtb_groupstats_destroy(self.h)
                self.h = c_void_p()
        except Exception:
            pass

    def gather(self, key: Column, cols: Sequence[int], miss_vals: Sequence[float], out_dtypes) -> List[torch.Tensor]:
        n = key.data.numel()
        codes = [dtype_code(d) for d in out_dtypes]
        outs = [torch.empty(n, dtype=_CODE2TORCH[c], device=key.data.device) for c in codes]
        _lib.check(self.lib.nvtb_groupstats_gather(
            self.h, _descs([key]), n, _lib.int_array(cols), len(cols), _lib.double_array(miss_vals),
            _lib.ptr_array([o.data_ptr() for o in outs]), _lib.int_array(codes), _lib.stream_ptr()))
        _count()
        return outs


# ------------------------------------------------------------------ session ops (csrc/groupby.cu)
AGG_SLOTS = ("count", "sum", "mean", "min", "max", "std", "var", "first", "last")


def _validity_buf(n: int, device) -> torch.Tensor:
    """a zeroed bitmask for n rows, padded to 32 bytes like pack_validity"""
    return torch.zeros(max((((n + 7) // 8 + 31) // 32) * 32, 32), dtype=torch.uint8, device=device)


def sort_rows(keys: Sequence[Column], descending: Optional[Sequence[bool]] = None, n_drop_null: int = 0):
    """stable row order by `keys` (first most significant), nulls of the first `n_drop_null` keys
    dropped, other nulls last (nvtb_sort_rows) -> (perm int32[n], kept-row count as a device
    int64[1]); the kept rows are perm[:n_kept]"""
    _lib.require_cuda()
    lib = _lib.load()
    n = _check_same_len(keys)
    dev = keys[0].data.device
    perm = torch.empty(n, dtype=torch.int32, device=dev)
    n_kept = torch.empty(1, dtype=torch.int64, device=dev)
    desc = [1 if d else 0 for d in (descending or [False] * len(keys))]
    with _timed("sort_rows", _in_bytes(keys) * 8):
        _lib.check(lib.nvtb_sort_rows(_descs(keys), _lib.int_array(desc), len(keys), int(n_drop_null), n,
                                      _ptr(perm), _ptr(n_kept), _lib.stream_ptr()))
    _count(4 + 8 * len(keys))
    return perm, n_kept


def segments(keys: Sequence[Column], perm: torch.Tensor, n_kept: torch.Tensor):
    """group boundaries of the sorted keys (nvtb_segments; synchronises) ->
    (offsets int64[n_groups + 1], n_groups, kept rows)"""
    lib = _lib.load()
    n = perm.numel()
    offsets = torch.empty(n + 1, dtype=torch.int64, device=perm.device)
    ng, nk = c_int64(0), c_int64(0)
    _lib.check(lib.nvtb_segments(_descs(keys), len(keys), _ptr(perm), n, _ptr(n_kept), _ptr(offsets),
                                 byref(ng), byref(nk), _lib.stream_ptr()))
    _count(4)
    return offsets[: ng.value + 1], ng.value, nk.value


def gather_rows(col: Column, perm: Optional[torch.Tensor], n: int, idx: Optional[torch.Tensor] = None,
                shift: int = 0) -> Column:
    """flat column rows col[perm[idx[i] + shift]] (nvtb_gather_rows); keeps the dictionary / bool flag"""
    lib = _lib.load()
    dev = col.data.device
    out = torch.empty(n, dtype=col.data.dtype, device=dev)
    valid = _validity_buf(n, dev) if col.validity is not None else None
    _lib.check(lib.nvtb_gather_rows(_descs([col]), _ptr(perm), _ptr(idx), int(shift), n, _ptr(out), _ptr(valid),
                                    _lib.stream_ptr()))
    _count()
    return Column(out, valid, None, col.dictionary, None, col.is_bool)


def segment_agg(col: Column, perm: torch.Tensor, offsets: torch.Tensor, n_groups: int, aggs: Sequence[str]):
    """{agg: Column} for aggs in AGG_SLOTS over every group (nvtb_segment_agg)"""
    lib = _lib.load()
    dev = col.data.device
    outs, valids, res = [None] * 9, [None] * 9, {}
    for a in aggs:
        s = AGG_SLOTS.index(a)
        dt = torch.int32 if a == "count" else torch.float32 if a in ("sum", "mean", "std", "var") else col.data.dtype
        outs[s] = torch.empty(n_groups, dtype=dt, device=dev)
        if a in ("mean", "min", "max", "std", "var") or (a in ("first", "last") and col.validity is not None):
            valids[s] = _validity_buf(n_groups, dev)
        keep_meta = a in ("min", "max", "first", "last")
        res[a] = Column(outs[s], valids[s], None, col.dictionary if keep_meta else None, None,
                        col.is_bool and keep_meta)
    with _timed("segment_agg", _in_bytes([col]) + 4.0 * perm.numel()):
        _lib.check(lib.nvtb_segment_agg(_descs([col]), _ptr(perm), _ptr(offsets), n_groups,
                                        _lib.ptr_array([o.data_ptr() if o is not None and o.numel() else None
                                                        for o in outs]),
                                        _lib.ptr_array([v.data_ptr() if v is not None else None for v in valids]),
                                        _lib.stream_ptr()))
    _count(6)
    return res


def segment_sorted_agg(col: Column, perm: torch.Tensor, offsets: torch.Tensor, n_groups: int, n_rows: int,
                       median=False, nunique=False):
    """{"median": Column, "nunique": Column} over groups in value order (nvtb_segment_sorted_agg)"""
    lib = _lib.load()
    dev = col.data.device
    res = {}
    med = torch.empty(n_groups, dtype=torch.float32, device=dev) if median else None
    med_v = _validity_buf(n_groups, dev) if median else None
    nun = torch.empty(n_groups, dtype=torch.int32, device=dev) if nunique else None
    _lib.check(lib.nvtb_segment_sorted_agg(_descs([col]), _ptr(perm), _ptr(offsets), n_groups, n_rows,
                                           _ptr(med) if median else None, _ptr(med_v) if median else None,
                                           _ptr(nun) if nunique else None, _lib.stream_ptr()))
    _count(4)
    if median:
        res["median"] = Column(med, med_v)
    if nunique:
        res["nunique"] = Column(nun)
    return res


def list_slice(col: Column, start: int, end: int, pad: bool = False, max_elements: int = 0, pad_value: float = 0.0,
               perm: Optional[torch.Tensor] = None, idx: Optional[torch.Tensor] = None, shift: int = 0,
               n_rows: Optional[int] = None) -> Column:
    """rows row[start:end] (Python slicing, padded to max_elements when `pad`) of a list column,
    optionally through a row permutation (nvtb_list_slice_offsets + nvtb_list_slice)"""
    _lib.require_cuda()
    lib = _lib.load()
    assert col.offsets is not None, "list_slice needs a list column"
    dev = col.data.device
    n = col.nrows if n_rows is None else n_rows
    offsets = torch.empty(n + 1, dtype=torch.int64, device=dev)
    total = c_int64(0)
    _lib.check(lib.nvtb_list_slice_offsets(_ptr(col.offsets), n, _ptr(perm), _ptr(idx), int(shift), int(start),
                                           int(end), 1 if pad else 0, int(max_elements), _ptr(offsets), byref(total),
                                           _lib.stream_ptr()))
    t = total.value
    leaves = torch.empty(t, dtype=col.data.dtype, device=dev)
    valid = _validity_buf(t, dev) if col.validity is not None else None
    with _timed("list_slice", 2.0 * t * col.data.element_size() + 16.0 * n):
        _lib.check(lib.nvtb_list_slice(_ptr(col.offsets), _descs([col]), n, _ptr(perm), _ptr(idx), int(shift),
                                       int(start), int(end), 1 if pad else 0, int(max_elements), float(pad_value),
                                       _ptr(offsets), t, _ptr(leaves), _ptr(valid), _lib.stream_ptr()))
    _count(4)
    return Column(leaves, valid, offsets, col.dictionary, None, col.is_bool)
