"""radix-sorting_b200 -- B200 (sm_100a) LSD radix sort behind the eloj/radix-sorting surface.

The product is ``librsx.so`` (hand-written CUDA + a C ABI, ``include/rsx.h``) and the C++
drop-in headers ``include/radix_sort.hpp`` / ``radix_sort_rank.hpp`` /
``radix_sort_basic_kdf.hpp``.  This module is the thin Python plumbing used by the tests and
``bench.py``: it binds the C ABI with ctypes and mirrors the reference's two entry points on
torch tensors (torch is used for device memory and streams only):

    radix_sort(src, aux, n=None, kf=None)            -> radix_sort.hpp:98-115
    radix_sort_rank(src, index_buffer, n=None, kf=None) -> radix_sort_rank.hpp:97-112
    radix_sort_segments / radix_sort_rank_segments        -> many independent arrays in one call

Both return the tensor / half that holds the result, like the reference returns a pointer.
There is NO CPU fallback: importing this module without a built ``librsx.so`` raises, and
every call on a machine without a CUDA device returns an error from the library.

The package directory name contains a hyphen (it is named after the reference repository);
import it with ``importlib.import_module("radix-sorting_b200")``.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import Optional

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RSX_LIB", os.path.join(HERE, "librsx.so"))  # RSX_LIB: A/B another build

KDF_UNSIGNED, KDF_SIGNED, KDF_FLOAT = 0, 1, 2
FLAG_INVERT = 1

RSX_OK = 0
RSX_ERR_INVALID, RSX_ERR_CUDA, RSX_ERR_NO_DEVICE = -1, -2, -3
RSX_ERR_WORKSPACE, RSX_ERR_IDX_RANGE, RSX_ERR_MIXED_MEMORY = -4, -5, -6

#: every symbol include/rsx.h declares (tests check that the library exports all of them)
EXPORTS = [
    "rsx_sort", "rsx_sort_rank", "rsx_sort_segments", "rsx_sort_rank_segments", "rsx_histogram", "rsx_histogram_column", "rsx_scatter_pass", "rsx_scatter_pass_to",
    "rsx_split_counts", "rsx_split_pass_to", "rsx_scatter_pass_append", "rsx_histogram_column_sampled", "rsx_sample_keys", "rsx_plan_compaction",
    "rsx_multi_route", "rsx_multi_splitters", "rsx_sort_shard", "rsx_sort_multi",
    "rsx_workspace_bytes",
    "rsx_reserve", "rsx_release", "rsx_fill_keys", "rsx_verify", "rsx_strerror",
    "rsx_last_cuda_error", "rsx_version", "rsx_total_kernel_launches", "rsx_set_option",
    "rsx_get_profile",
]


class RsxLayout(C.Structure):
    """struct rsx_layout (include/rsx.h)."""
    _fields_ = [("record_bytes", C.c_uint32), ("key_offset", C.c_uint32),
                ("key_bytes", C.c_uint32), ("kdf_kind", C.c_uint32), ("flags", C.c_uint32)]


class RsxReport(C.Structure):
    """struct rsx_report (include/rsx.h)."""
    _fields_ = [("early_exit", C.c_uint32), ("ncols", C.c_uint32), ("live_mask", C.c_uint32),
                ("result_in_aux", C.c_uint32), ("kernel_launches", C.c_uint32),
                ("staged", C.c_uint32), ("compacted_passes", C.c_uint32)]


RSX_MAX_RANKS = 16
MULTI_NO_FUSED, MULTI_NO_KEY_RANGE, MULTI_FULL_HISTOGRAM, MULTI_EXACT = 1, 2, 4, 8

ALLGATHER_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t)
BARRIER_FN = C.CFUNCTYPE(C.c_int, C.c_void_p)
ALLTOALLV_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p, C.POINTER(C.c_uint64))


class RsxComm(C.Structure):
    """struct rsx_comm (include/rsx.h): the two collectives rsx_sort_shard needs, as callbacks."""
    _fields_ = [("rank", C.c_int), ("world", C.c_int), ("allgather", ALLGATHER_FN), ("barrier", BARRIER_FN),
                ("alltoallv", ALLTOALLV_FN), ("ctx", C.c_void_p)]


_LP = C.POINTER(RsxLayout)
OPS_HIST_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, _LP, C.POINTER(C.c_uint64), C.c_void_p)
OPS_SAMPLE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, _LP, C.c_size_t, C.POINTER(C.c_uint64), C.c_void_p)
OPS_SPLIT_COUNTS_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, _LP, C.POINTER(C.c_uint64), C.c_int,
                                  C.POINTER(C.c_uint64), C.c_void_p)
OPS_PARTITION_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, _LP, C.c_int, C.POINTER(C.c_uint8),
                               C.POINTER(C.c_uint64), C.c_int, C.POINTER(C.c_uint64), C.c_int, C.c_void_p)
OPS_HIST_COLUMN_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, _LP, C.c_int, C.POINTER(C.c_uint64), C.c_void_p)
OPS_SORT_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, _LP, C.POINTER(C.c_void_p), C.c_void_p)


class RsxShardOps(C.Structure):
    """struct rsx_shard_ops: local primitives (NULL pointer = the library's CUDA kernels)."""
    _fields_ = [("hist", OPS_HIST_FN), ("sample", OPS_SAMPLE_FN), ("split_counts", OPS_SPLIT_COUNTS_FN),
                ("partition_to", OPS_PARTITION_FN), ("sort", OPS_SORT_FN), ("ctx", C.c_void_p),
                ("hist_column", OPS_HIST_COLUMN_FN)]


class RsxRoute(C.Structure):
    """struct rsx_route."""
    _fields_ = [("routing_column", C.c_int32), ("live_mask", C.c_uint32), ("key_range", C.c_uint32), ("pad", C.c_uint32),
                ("owner", C.c_uint8 * 256), ("n_in", C.c_uint64 * RSX_MAX_RANKS), ("send_counts", C.c_uint64 * RSX_MAX_RANKS),
                ("recv_counts", C.c_uint64 * RSX_MAX_RANKS), ("dest_offset", C.c_uint64 * RSX_MAX_RANKS),
                ("n_out", C.c_uint64), ("max_n_out", C.c_uint64), ("n_total", C.c_uint64), ("imbalance", C.c_double)]


class RsxMultiReport(C.Structure):
    """struct rsx_multi_report."""
    _fields_ = [("routing_column", C.c_int32), ("key_range", C.c_uint32), ("live_mask", C.c_uint32), ("fused", C.c_uint32),
                ("append", C.c_uint32), ("pad", C.c_uint32), ("n_total", C.c_uint64), ("needed_capacity", C.c_uint64), ("imbalance", C.c_double),
                ("seconds_histogram", C.c_double), ("seconds_routing", C.c_double), ("seconds_exchange", C.c_double),
                ("seconds_local_sort", C.c_double)]


class RsxError(RuntimeError):
    def __init__(self, status: int, where: str):
        self.status = status
        lib = _lib()
        msg = lib.rsx_strerror(status).decode()
        detail = lib.rsx_last_cuda_error().decode()
        super().__init__(f"{where}: {msg} [{status}]" + (f" -- {detail}" if detail and status == RSX_ERR_CUDA else ""))


_LIB = None


def _lib() -> C.CDLL:
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C radix-sorting_b200/csrc`).  There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, sz, u64p = C.c_void_p, C.c_size_t, C.POINTER(C.c_uint64)
    LP, RP = C.POINTER(RsxLayout), C.POINTER(RsxReport)
    L.rsx_sort.restype = C.c_int
    L.rsx_sort.argtypes = [vp, vp, sz, LP, C.POINTER(vp), RP, vp]
    L.rsx_sort_rank.restype = C.c_int
    L.rsx_sort_rank.argtypes = [vp, vp, sz, LP, C.c_int, C.POINTER(vp), RP, vp]
    L.rsx_sort_segments.restype = C.c_int
    L.rsx_sort_segments.argtypes = [vp, vp, sz, u64p, sz, LP, C.POINTER(vp), RP, vp]
    L.rsx_sort_rank_segments.restype = C.c_int
    L.rsx_sort_rank_segments.argtypes = [vp, vp, sz, u64p, sz, LP, C.c_int, C.POINTER(vp), RP, vp]
    L.rsx_histogram.restype = C.c_int
    L.rsx_histogram.argtypes = [vp, sz, LP, u64p, u64p, RP, vp]
    L.rsx_histogram_column.restype = C.c_int
    L.rsx_histogram_column.argtypes = [vp, sz, LP, C.c_int, u64p, vp]
    L.rsx_scatter_pass.restype = C.c_int
    L.rsx_scatter_pass.argtypes = [vp, vp, vp, vp, C.c_int, sz, LP, C.c_int, vp]
    if hasattr(L, "rsx_scatter_pass_to"):
        L.rsx_scatter_pass_to.restype = C.c_int
        L.rsx_scatter_pass_to.argtypes = [vp, sz, LP, C.c_int, C.POINTER(C.c_uint8), u64p, C.c_int, vp]
    if hasattr(L, "rsx_split_counts"):  # absent only in older builds loaded through RSX_LIB for A/B runs
        L.rsx_split_counts.restype = C.c_int
        L.rsx_split_counts.argtypes = [vp, sz, LP, u64p, C.c_int, u64p, vp]
        L.rsx_split_pass_to.restype = C.c_int
        L.rsx_split_pass_to.argtypes = [vp, sz, LP, u64p, C.c_int, u64p, vp]
    L.rsx_scatter_pass_append.restype = C.c_int
    L.rsx_scatter_pass_append.argtypes = [vp, sz, LP, C.c_int, C.POINTER(C.c_uint8), u64p, C.c_int, u64p, u64p, u64p, C.c_int,
                                          C.POINTER(C.c_uint32), vp]
    L.rsx_histogram_column_sampled.restype = C.c_int
    L.rsx_histogram_column_sampled.argtypes = [vp, sz, LP, C.c_int, sz, u64p, vp]
    L.rsx_sample_keys.restype = C.c_int
    L.rsx_sample_keys.argtypes = [vp, sz, LP, sz, u64p, vp]
    L.rsx_plan_compaction.restype = C.c_int
    L.rsx_plan_compaction.argtypes = [C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.POINTER(C.c_uint32), u64p]
    L.rsx_multi_route.restype = C.c_int
    L.rsx_multi_route.argtypes = [u64p, C.c_int, C.c_int, C.c_int, C.c_double, C.POINTER(RsxRoute)]
    L.rsx_multi_splitters.restype = C.c_int
    L.rsx_multi_splitters.argtypes = [u64p, sz, C.c_int, u64p]
    L.rsx_sort_shard.restype = C.c_int
    L.rsx_sort_shard.argtypes = [C.POINTER(RsxComm), C.POINTER(RsxShardOps), vp, sz, vp, C.POINTER(vp), sz, LP, C.c_uint32,
                                 C.POINTER(vp), C.POINTER(sz), C.POINTER(RsxMultiReport), vp]
    L.rsx_sort_multi.restype = C.c_int
    L.rsx_sort_multi.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(vp), C.POINTER(vp), C.POINTER(sz), sz, LP,
                                 C.c_uint32, C.POINTER(vp), C.POINTER(sz), C.POINTER(RsxMultiReport)]
    L.rsx_workspace_bytes.restype = sz
    L.rsx_workspace_bytes.argtypes = [sz, LP, C.c_int]
    L.rsx_reserve.restype = C.c_int
    L.rsx_reserve.argtypes = [sz]
    L.rsx_release.restype = None
    L.rsx_release.argtypes = []
    L.rsx_fill_keys.restype = C.c_int
    L.rsx_fill_keys.argtypes = [vp, sz, C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.c_uint64,
                                C.c_uint64, vp]
    L.rsx_verify.restype = C.c_int
    L.rsx_verify.argtypes = [vp, sz, LP, u64p, u64p, u64p, vp]
    L.rsx_strerror.restype = C.c_char_p
    L.rsx_strerror.argtypes = [C.c_int]
    L.rsx_last_cuda_error.restype = C.c_char_p
    L.rsx_last_cuda_error.argtypes = []
    L.rsx_version.restype = C.c_int
    L.rsx_version.argtypes = []
    L.rsx_total_kernel_launches.restype = C.c_uint64
    L.rsx_total_kernel_launches.argtypes = []
    L.rsx_set_option.restype = C.c_int
    L.rsx_set_option.argtypes = [C.c_char_p, C.c_long]
    L.rsx_get_profile.restype = C.c_int
    L.rsx_get_profile.argtypes = [C.POINTER(C.c_float), C.c_int]
    _LIB = L
    return L


def lib() -> C.CDLL:
    """The loaded C-ABI library (raises ImportError if it was never built)."""
    return _lib()


# ---- key-derivation descriptors: the KeyFunc of radix_sort.hpp:31-35 across a C ABI ------------

@dataclass(frozen=True)
class KeyFunc:
    """Describes `kf`: where the key sits in the record and how it is derived.

    kind: KDF_UNSIGNED (radix_sort_basic_kdf.hpp:19-23), KDF_SIGNED (:26-30), KDF_FLOAT (:32-46)
    descending: complement the derived key (README.md:564-574)
    record_bytes/key_offset/key_bytes: None = the whole element is the key
    """
    kind: int
    descending: bool = False
    record_bytes: Optional[int] = None
    key_offset: int = 0
    key_bytes: Optional[int] = None

    def layout(self, elem_bytes: int) -> RsxLayout:
        rb = self.record_bytes or elem_bytes
        kb = self.key_bytes or rb
        return RsxLayout(rb, self.key_offset, kb, self.kind, FLAG_INVERT if self.descending else 0)


def _torch():
    import torch
    return torch


def default_kdf(dtype, descending: bool = False) -> KeyFunc:
    """basic_kdfs::kdf overload resolution by element type (radix_sort_basic_kdf.hpp:19-46)."""
    torch = _torch()
    if dtype == torch.bool:
        raise TypeError("bool keys are excluded by the reference (radix_sort_basic_kdf.hpp:20,27)")
    if dtype.is_floating_point:
        if dtype not in (torch.float32, torch.float64):
            raise TypeError(f"no KDF for {dtype}: the reference ships float and double only")
        return KeyFunc(KDF_FLOAT, descending)
    signed = dtype in (torch.int8, torch.int16, torch.int32, torch.int64)
    return KeyFunc(KDF_SIGNED if signed else KDF_UNSIGNED, descending)


def _stream_ptr(t) -> int:
    torch = _torch()
    return torch.cuda.current_stream(t.device).cuda_stream if t.is_cuda else 0


def _check(t, name: str):
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")


def radix_sort(src, aux, n: Optional[int] = None, kf: Optional[KeyFunc] = None, *,
               report: Optional[RsxReport] = None):
    """T* radix_sort(T* src, T* aux, size_t n, KeyFunc&& kf)  -- radix_sort.hpp:98-115.

    `src`/`aux`: torch tensors of the same dtype (device tensors are sorted on the GPU in place;
    CPU tensors are staged).  For records pass uint8 tensors (or any dtype) plus a KeyFunc with
    record_bytes.  Returns `src` or `aux`, whichever holds the sorted data (both are clobbered).
    """
    torch = _torch()
    _check(src, "src"), _check(aux, "aux")
    if src.dtype != aux.dtype or src.device != aux.device:
        raise ValueError("src and aux must have the same dtype and device")
    kf = kf or default_kdf(src.dtype)
    L = kf.layout(src.element_size())
    count = src.numel() * src.element_size() // L.record_bytes
    n = count if n is None else n
    if n > count or aux.numel() * aux.element_size() < n * L.record_bytes:
        raise ValueError("n exceeds the buffers")
    res = C.c_void_p()
    rep = report if report is not None else RsxReport()
    if src.is_cuda:
        with torch.cuda.device(src.device):
            st = _lib().rsx_sort(src.data_ptr(), aux.data_ptr(), n, C.byref(L), C.byref(res),
                                 C.byref(rep), _stream_ptr(src))
    else:
        st = _lib().rsx_sort(src.data_ptr(), aux.data_ptr(), n, C.byref(L), C.byref(res),
                             C.byref(rep), 0)
    if st != RSX_OK:
        raise RsxError(st, "rsx_sort")
    return aux if (n and res.value == aux.data_ptr() and res.value != src.data_ptr()) else src


def radix_sort_rank(src, index_buffer, n: Optional[int] = None, kf: Optional[KeyFunc] = None, *,
                    report: Optional[RsxReport] = None):
    """IdxType* radix_sort_rank(const T* src, IdxType* index_buffer, size_t n, KeyFunc&& kf)
    -- radix_sort_rank.hpp:97-112.  `index_buffer` has 2n entries (README.md:520-526); returns
    the n-entry half that holds the ranks.  `src` is not modified."""
    torch = _torch()
    _check(src, "src"), _check(index_buffer, "index_buffer")
    if src.device != index_buffer.device:
        raise ValueError("src and index_buffer must be on the same device")
    kf = kf or default_kdf(src.dtype)
    L = kf.layout(src.element_size())
    count = src.numel() * src.element_size() // L.record_bytes
    n = count if n is None else n
    if n > count or index_buffer.numel() < 2 * n:
        raise ValueError("index_buffer must hold 2n entries")
    ib_bytes = index_buffer.element_size()
    res = C.c_void_p()
    rep = report if report is not None else RsxReport()
    if src.is_cuda:
        with torch.cuda.device(src.device):
            st = _lib().rsx_sort_rank(src.data_ptr(), index_buffer.data_ptr(), n, C.byref(L), ib_bytes,
                                      C.byref(res), C.byref(rep), _stream_ptr(src))
    else:
        st = _lib().rsx_sort_rank(src.data_ptr(), index_buffer.data_ptr(), n, C.byref(L), ib_bytes,
                                  C.byref(res), C.byref(rep), 0)
    if st != RSX_OK:
        raise RsxError(st, "rsx_sort_rank")
    flat = index_buffer.view(-1)
    off = (res.value - index_buffer.data_ptr()) // ib_bytes if n else 0
    return flat[off:off + n]


def _offsets(offsets):
    """offsets (int64 tensor on the CPU or a device, or a sequence of ints) -> (pointer, nseg, keep-alive)."""
    torch = _torch()
    if not isinstance(offsets, torch.Tensor):
        offsets = torch.tensor([int(x) for x in offsets], dtype=torch.int64)
    if offsets.dtype not in (torch.int64, torch.uint64) or offsets.dim() != 1 or offsets.numel() < 1:
        raise ValueError("offsets must be a 1-D int64 tensor or a sequence of nseg + 1 ints")
    offsets = offsets.contiguous()
    return C.cast(C.c_void_p(offsets.data_ptr()), C.POINTER(C.c_uint64)), offsets.numel() - 1, offsets


def radix_sort_segments(src, aux, offsets, kf: Optional[KeyFunc] = None, *, report: Optional[RsxReport] = None):
    """Sorts every segment [offsets[s], offsets[s+1]) of `src` independently, in one call
    (rsx_sort_segments).  `src`/`aux`: device tensors of the same dtype, n = offsets[-1] records
    each; `offsets`: int64 tensor (CPU or CUDA) or a sequence of nseg + 1 ints.  Returns `src` or
    `aux`, whichever holds the whole sorted batch (the reference's parity rule over the batch)."""
    torch = _torch()
    _check(src, "src"), _check(aux, "aux")
    if src.dtype != aux.dtype or src.device != aux.device:
        raise ValueError("src and aux must have the same dtype and device")
    kf = kf or default_kdf(src.dtype)
    L = kf.layout(src.element_size())
    count = src.numel() * src.element_size() // L.record_bytes
    off, nseg, keep = _offsets(offsets)
    n = int(keep[-1])
    if n > count or aux.numel() * aux.element_size() < n * L.record_bytes:
        raise ValueError("offsets[-1] exceeds the buffers")
    res = C.c_void_p()
    rep = report if report is not None else RsxReport()
    with torch.cuda.device(src.device if src.is_cuda else None):
        st = _lib().rsx_sort_segments(src.data_ptr(), aux.data_ptr(), n, off, nseg, C.byref(L), C.byref(res),
                                      C.byref(rep), _stream_ptr(src))
    if st != RSX_OK:
        raise RsxError(st, "rsx_sort_segments")
    return aux if (n and res.value == aux.data_ptr() and res.value != src.data_ptr()) else src


def radix_sort_rank_segments(src, index_buffer, offsets, kf: Optional[KeyFunc] = None, *,
                             report: Optional[RsxReport] = None):
    """Segment-relative stable argsort of every segment of `src` in one call (rsx_sort_rank_segments).
    `index_buffer` has 2n entries; returns the n-entry half that holds the ranks.  `src` is not
    modified."""
    torch = _torch()
    _check(src, "src"), _check(index_buffer, "index_buffer")
    if src.device != index_buffer.device:
        raise ValueError("src and index_buffer must be on the same device")
    kf = kf or default_kdf(src.dtype)
    L = kf.layout(src.element_size())
    count = src.numel() * src.element_size() // L.record_bytes
    off, nseg, keep = _offsets(offsets)
    n = int(keep[-1])
    if n > count or index_buffer.numel() < 2 * n:
        raise ValueError("index_buffer must hold 2n entries")
    ib_bytes = index_buffer.element_size()
    res = C.c_void_p()
    rep = report if report is not None else RsxReport()
    with torch.cuda.device(src.device if src.is_cuda else None):
        st = _lib().rsx_sort_rank_segments(src.data_ptr(), index_buffer.data_ptr(), n, off, nseg, C.byref(L), ib_bytes,
                                           C.byref(res), C.byref(rep), _stream_ptr(src))
    if st != RSX_OK:
        raise RsxError(st, "rsx_sort_rank_segments")
    off_el = (res.value - index_buffer.data_ptr()) // ib_bytes if n else 0
    return index_buffer.view(-1)[off_el:off_el + n]


def histogram(src, kf: Optional[KeyFunc] = None):
    """Phases 1-3 of rs_sort_main (radix_sort.hpp:46-80) on the device.
    Returns (hist[key_bytes,256] uint64 numpy, descents, RsxReport)."""
    import numpy as np
    torch = _torch()
    kf = kf or default_kdf(src.dtype)
    L = kf.layout(src.element_size())
    n = src.numel() * src.element_size() // L.record_bytes
    hist = np.zeros((L.key_bytes, 256), dtype=np.uint64)
    desc = C.c_uint64(0)
    rep = RsxReport()
    with torch.cuda.device(src.device):
        st = _lib().rsx_histogram(src.data_ptr(), n, C.byref(L),
                                  hist.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(desc),
                                  C.byref(rep), _stream_ptr(src))
    if st != RSX_OK:
        raise RsxError(st, "rsx_histogram")
    return hist, int(desc.value), rep


def scatter_pass(src, dst, col: int, kf: Optional[KeyFunc] = None, payload_src=None, payload_dst=None):
    """One stable counting-sort pass on column `col` (radix_sort.hpp:83-88)."""
    torch = _torch()
    kf = kf or default_kdf(src.dtype)
    L = kf.layout(src.element_size())
    n = src.numel() * src.element_size() // L.record_bytes
    pb = payload_src.element_size() if payload_src is not None else 0
    with torch.cuda.device(src.device):
        st = _lib().rsx_scatter_pass(src.data_ptr(), dst.data_ptr(),
                                     payload_src.data_ptr() if pb else None,
                                     payload_dst.data_ptr() if pb else None,
                                     pb, n, C.byref(L), col, _stream_ptr(src))
    if st != RSX_OK:
        raise RsxError(st, "rsx_scatter_pass")
    return dst


def scatter_pass_to(src, col: int, owner, dest_base, kf: Optional[KeyFunc] = None):
    """Fused partition + exchange: stable pass on `col` whose buckets go to destination
    owner[bucket] (256 ints, non-decreasing); every tile appends one contiguous run per
    destination at byte address dest_base[D] (typically peer-GPU memory)."""
    torch = _torch()
    kf = kf or default_kdf(src.dtype)
    L = kf.layout(src.element_size())
    n = src.numel() * src.element_size() // L.record_bytes
    own = (C.c_uint8 * 256)(*[int(x) for x in owner])
    base = (C.c_uint64 * len(dest_base))(*[int(x) for x in dest_base])
    with torch.cuda.device(src.device):
        st = _lib().rsx_scatter_pass_to(src.data_ptr(), n, C.byref(L), col, own, base, len(dest_base),
                                        _stream_ptr(src))
    if st != RSX_OK:
        raise RsxError(st, "rsx_scatter_pass_to")


def split_counts(src, splitters, kf: Optional[KeyFunc] = None):
    """Records per key range: range index = number of (ascending, derived-key) splitters <= key."""
    torch = _torch()
    kf = kf or default_kdf(src.dtype)
    L = kf.layout(src.element_size())
    n = src.numel() * src.element_size() // L.record_bytes
    sp = (C.c_uint64 * len(splitters))(*[int(x) for x in splitters])
    out = (C.c_uint64 * (len(splitters) + 1))()
    with torch.cuda.device(src.device):
        st = _lib().rsx_split_counts(src.data_ptr(), n, C.byref(L), sp, len(splitters), out, _stream_ptr(src))
    if st != RSX_OK:
        raise RsxError(st, "rsx_split_counts")
    return [int(x) for x in out]


def split_pass_to(src, splitters, dest_base, kf: Optional[KeyFunc] = None):
    """Stable partition by key range; range D is appended at byte address dest_base[D]."""
    torch = _torch()
    kf = kf or default_kdf(src.dtype)
    L = kf.layout(src.element_size())
    n = src.numel() * src.element_size() // L.record_bytes
    sp = (C.c_uint64 * len(splitters))(*[int(x) for x in splitters])
    base = (C.c_uint64 * len(dest_base))(*[int(x) for x in dest_base])
    assert len(dest_base) == len(splitters) + 1
    with torch.cuda.device(src.device):
        st = _lib().rsx_split_pass_to(src.data_ptr(), n, C.byref(L), sp, len(splitters), base, _stream_ptr(src))
    if st != RSX_OK:
        raise RsxError(st, "rsx_split_pass_to")


def fill_keys(dst, seed: int, start: int = 0, dist: str = "uniform", mask: int = (1 << 64) - 1,
              orv: int = 0):
    """Device twin of keygen.fill: writes dst.numel() keys of dst.element_size() bytes."""
    from .keygen import DIST_CODE
    torch = _torch()
    with torch.cuda.device(dst.device):
        st = _lib().rsx_fill_keys(dst.data_ptr(), dst.numel(), dst.element_size(), seed, start,
                                  DIST_CODE[dist], mask, orv, _stream_ptr(dst))
    if st != RSX_OK:
        raise RsxError(st, "rsx_fill_keys")
    return dst


def verify(data, kf: Optional[KeyFunc] = None, n: Optional[int] = None):
    """On-device order + multiset check: returns (descents, checksum_sum, checksum_xor)."""
    torch = _torch()
    kf = kf or default_kdf(data.dtype)
    L = kf.layout(data.element_size())
    count = data.numel() * data.element_size() // L.record_bytes
    n = count if n is None else n
    d, s, x = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
    with torch.cuda.device(data.device):
        st = _lib().rsx_verify(data.data_ptr(), n, C.byref(L), C.byref(d), C.byref(s), C.byref(x),
                               _stream_ptr(data))
    if st != RSX_OK:
        raise RsxError(st, "rsx_verify")
    return int(d.value), int(s.value), int(x.value)


def reserve(nbytes: int) -> None:
    st = _lib().rsx_reserve(nbytes)
    if st != RSX_OK:
        raise RsxError(st, "rsx_reserve")


def workspace_bytes(n: int, layout: RsxLayout, rank_idx_bytes: int = 0) -> int:
    return int(_lib().rsx_workspace_bytes(n, C.byref(layout), rank_idx_bytes))


def set_profile(on: bool) -> None:
    _lib().rsx_set_option(b"profile", 1 if on else 0)


def get_profile():
    """Per-kernel device ms of the last profiled sort: [K1, K2, pass col0, pass col1, ...]."""
    buf = (C.c_float * 16)()
    k = _lib().rsx_get_profile(buf, 16)
    return [float(buf[i]) for i in range(max(k, 0))]


def total_kernel_launches() -> int:
    return int(_lib().rsx_total_kernel_launches())


_lib()  # fail loudly at import time if the CUDA library is missing
