"""Python-side call wrappers around the C ABI (device tensors in, device tensors out).

One function per ABI entry point (include/sparse_b200.h); each cites the reference closure it
replaces.  Everything here launches CUDA kernels from libsparse_b200.so on torch's current stream;
torch is used only to own the device allocations.
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _device as D
from . import _lib
from ._lib import i32, i64, vp


def _t():
    return D.torch()


def _idx_bytes(t) -> int:
    return 8 if t.dtype == _t().int64 else 4


def _esize(t) -> int:
    return t.element_size()


def _sp():
    return vp(D.stream_ptr())


def _i64arr(vals):
    arr = (ctypes.c_int64 * max(len(vals), 1))(*[int(v) for v in vals])
    return arr


def _i32arr(vals):
    arr = (ctypes.c_int32 * max(len(vals), 1))(*[int(v) for v in vals])
    return arr


def _scalar_bytes(value, dtype) -> ctypes.Array:
    """16-byte host buffer holding `value` as `dtype` (for fill values / scalars; complex128 is the widest)."""
    a = np.zeros(1, dtype=np.dtype(dtype))
    a[0] = value
    buf = (ctypes.c_uint8 * 16)()
    ctypes.memmove(buf, a.ctypes.data, a.itemsize)
    return buf


def empty(n, dtype, like=None):
    t = _t()
    dev = like.device if like is not None else D.device()
    return t.empty(n, dtype=dtype if isinstance(dtype, t.dtype) else D.torch_dtype(dtype), device=dev)


# ------------------------------------------------------------------------------------------------
# K1
# ------------------------------------------------------------------------------------------------
def spmm_csr_dense(a_data, a_indices, a_indptr, b, M: int, K: int, N: int, out=None, *, n_panels=1,
                   rows_sorted=None, long_rows=False):
    """out[M,N] = CSR(A) @ B -- replaces _dot_csr_ndarray (_common.py:720-755).

    All arguments are CUDA tensors; `b` is (K, N) row-major (row stride may exceed N).
    Bit-identical to the reference loop (stored order, unfused multiply/add).
    n_panels: 1 = one-pass kernel; >= 2 = column-panel passes (L2-resident slices of B; needs rows sorted by
    column); 0 = let the library choose from the size of B and nnz / M.
    """
    lib = _lib.load()
    t = _t()
    dt = D.np_dtype(a_data)
    assert b.dtype == a_data.dtype, "promote operands to _dot_dtype first"
    assert a_indices.dtype == a_indptr.dtype
    if b.dim() != 2 or (N > 1 and b.stride(1) != 1):
        b = b.contiguous()
    if out is None:
        out = t.empty((M, N), dtype=a_data.dtype, device=a_data.device)
    ldb = b.stride(0) if K > 1 else max(N, 1)
    ldc = out.stride(0) if M > 1 else max(N, 1)
    if n_panels != 1 and rows_sorted is None:
        rows_sorted = csr_rows_sorted(a_indices, a_indptr, M)
    rc = lib.b2s_spmm_csr_dense_ex(
        i32(D.dtype_code(dt)), i32(_idx_bytes(a_indices)), i64(M), i64(K), i64(N), i64(a_data.shape[0]),
        vp(D.ptr(a_data)), vp(D.ptr(a_indices)), vp(D.ptr(a_indptr)), vp(D.ptr(b)), i64(max(ldb, N)), vp(D.ptr(out)),
        i64(max(ldc, N)), i32(n_panels if (n_panels == 1 or rows_sorted) else 1), i32(1 if rows_sorted else 0),
        i32(1 if long_rows else 0), _sp(),
    )
    _lib.check(rc, "b2s_spmm_csr_dense_ex")
    return out


def csr_max_row_nnz(a_indptr, M) -> int:
    """Largest row length of a CSR (one device reduction + sync)."""
    r = ctypes.c_int64(0)
    _lib.check(_lib.load().b2s_csr_max_row_nnz(i32(_idx_bytes(a_indptr)), i64(M), vp(D.ptr(a_indptr)), ctypes.byref(r),
                                               _sp()))
    return int(r.value)


def csr_rows_sorted(a_indices, a_indptr, M) -> bool:
    """True when every CSR row has non-decreasing column indices (precondition of the panel passes)."""
    r = ctypes.c_int(1)
    _lib.check(_lib.load().b2s_csr_rows_sorted(i32(_idx_bytes(a_indices)), i64(M), vp(D.ptr(a_indptr)),
                                               vp(D.ptr(a_indices)), ctypes.byref(r), _sp()))
    return bool(r.value)


def spmm_csr_dense_host(a_data: np.ndarray, a_indices: np.ndarray, a_indptr: np.ndarray, b: np.ndarray,
                        out: np.ndarray | None = None) -> np.ndarray:
    """Host-buffer form of K1 (H2D + kernel + D2H inside the call)."""
    _lib.require_device()
    lib = _lib.load()
    dt = a_data.dtype
    assert b.dtype == dt
    M = len(a_indptr) - 1
    K, N = b.shape
    idt = np.int32 if (a_indices.dtype == np.int32 and a_indptr.dtype == np.int32) else np.int64
    a_indices = np.ascontiguousarray(a_indices, dtype=idt)
    a_indptr = np.ascontiguousarray(a_indptr, dtype=idt)
    b = np.ascontiguousarray(b)
    if out is None:
        out = np.empty((M, N), dtype=dt)
    rc = lib.b2s_spmm_csr_dense_host(
        i32(D.dtype_code(dt)), i32(np.dtype(idt).itemsize), i64(M), i64(K), i64(N), i64(len(a_data)),
        vp(a_data.ctypes.data), vp(a_indices.ctypes.data), vp(a_indptr.ctypes.data), vp(b.ctypes.data),
        vp(out.ctypes.data),
    )
    _lib.check(rc, "b2s_spmm_csr_dense_host")
    return out


def spmm_set_variant(variant: int = 1, unroll: int = 8):
    _lib.check(_lib.load().b2s_spmm_set_variant(i32(variant), i32(unroll)))


def spmm_host_set_threads(n: int = -1):
    """Host threads narrowing int64 indices before the upload of the host-buffer product (-1 auto, 0 device-side)."""
    _lib.check(_lib.load().b2s_spmm_host_set_threads(i32(n)))


def spmm_host_set_pipeline(chunks: int = 16, slots: int = 4):
    _lib.check(_lib.load().b2s_spmm_host_set_pipeline(i32(chunks), i32(slots)))


def host_narrow(src: np.ndarray, dst: np.ndarray):
    """dst[i] = int32(src[i]) on the host thread pool of the library (both C-contiguous host arrays)."""
    assert src.dtype == np.int64 and dst.dtype == np.int32 and src.size == dst.size
    _lib.check(_lib.load().b2s_host_narrow_i64_i32(vp(src.ctypes.data), vp(dst.ctypes.data), i64(src.size)))
    return dst


# ------------------------------------------------------------------------------------------------
# prims
# ------------------------------------------------------------------------------------------------
def linearize(coords, strides):
    """keys[i] = sum_d coords[d, i] * strides[d]  (linear_loc, _coo/common.py:56-64, with permutation)."""
    t = _t()
    ndim, nnz = coords.shape
    keys = t.empty(nnz, dtype=t.int64, device=coords.device)
    if nnz == 0 or ndim == 0:
        return keys.zero_() if nnz else keys
    if coords.stride(1) != 1:
        coords = coords.contiguous()
    rc = _lib.load().b2s_coo_linearize(i32(_idx_bytes(coords)), i32(ndim), i64(nnz), vp(D.ptr(coords)),
                                      i64(coords.stride(0)), _i64arr(strides), vp(D.ptr(keys)), _sp())
    _lib.check(rc, "b2s_coo_linearize")
    return keys


def diag_flags(coords, first):
    """uint8 flags: entry i kept iff coords[d, i] == coords[first[d], i] for all d (einsum trace selector)."""
    t = _t()
    ndim, nnz = coords.shape
    flags = t.empty(nnz, dtype=t.uint8, device=coords.device)
    if nnz == 0:
        return flags
    if coords.stride(1) != 1:
        coords = coords.contiguous()
    rc = _lib.load().b2s_coo_diag_flags(i32(_idx_bytes(coords)), i32(ndim), i64(nnz), vp(D.ptr(coords)),
                                        i64(coords.stride(0)), _i32arr(first), vp(D.ptr(flags)), _sp())
    _lib.check(rc, "b2s_coo_diag_flags")
    return flags


def slice_keys(keys, shape, start, step, count, out_stride):
    """(flags, new keys) of basic indexing: axis d keeps c = start[d] + j*step[d], 0 <= j < count[d]."""
    t = _t()
    n = keys.shape[0]
    flags = t.empty(n, dtype=t.uint8, device=keys.device)
    okeys = t.empty(n, dtype=t.int64, device=keys.device)
    if n:
        rc = _lib.load().b2s_coo_slice_keys(i32(len(shape)), i64(n), vp(D.ptr(keys)), _i64arr(shape), _i64arr(start),
                                            _i64arr(step), _i64arr(count), _i64arr(out_stride), vp(D.ptr(flags)),
                                            vp(D.ptr(okeys)), _sp())
        _lib.check(rc, "b2s_coo_slice_keys")
    return flags, okeys


def unravel(keys, shape, idx_dtype=np.int64):
    """coords[ndim, nnz] of C-order linear `keys` over `shape`."""
    t = _t()
    ndim, nnz = len(shape), keys.shape[0]
    coords = t.empty((ndim, nnz), dtype=D.torch_dtype(idx_dtype), device=keys.device)
    if nnz == 0 or ndim == 0:
        return coords
    rc = _lib.load().b2s_coo_unravel(i32(np.dtype(idx_dtype).itemsize), i32(ndim), i64(nnz), vp(D.ptr(keys)),
                                    _i64arr(shape), vp(D.ptr(coords)), i64(coords.stride(0)), _sp())
    _lib.check(rc, "b2s_coo_unravel")
    return coords


def keys_flags(keys):
    """(unsorted, has_duplicates) -- COO._sort_indices / _sum_duplicates tests (_coo/core.py:1310-1343)."""
    a, b = ctypes.c_int(0), ctypes.c_int(0)
    rc = _lib.load().b2s_keys_flags(vp(D.ptr(keys)), i64(keys.shape[0]), ctypes.byref(a), ctypes.byref(b), _sp())
    _lib.check(rc, "b2s_keys_flags")
    return bool(a.value), bool(b.value)


def sort_keys(keys, key_bits=64):
    """Stable argsort: returns (sorted_keys, perm)."""
    t = _t()
    n = keys.shape[0]
    out = t.empty_like(keys)
    perm = t.empty(n, dtype=t.int64, device=keys.device)
    rc = _lib.load().b2s_sort_keys(vp(D.ptr(keys)), i64(n), i32(key_bits), vp(D.ptr(out)), vp(D.ptr(perm)), _sp())
    _lib.check(rc, "b2s_sort_keys")
    return out, perm


def gather(x, perm):
    t = _t()
    out = t.empty(perm.shape[0], dtype=x.dtype, device=x.device)
    rc = _lib.load().b2s_gather(i32(_esize(x)), vp(D.ptr(x)), vp(D.ptr(perm)), i64(perm.shape[0]), vp(D.ptr(out)),
                               _sp())
    _lib.check(rc, "b2s_gather")
    return out


def gather_rows(x2d, perm):
    """x2d[:, perm] for a [rows, n] tensor."""
    t = _t()
    out = t.empty((x2d.shape[0], perm.shape[0]), dtype=x2d.dtype, device=x2d.device)
    for d in range(x2d.shape[0]):
        row = x2d[d]
        if row.stride(0) != 1:
            row = row.contiguous()
        rc = _lib.load().b2s_gather(i32(_esize(x2d)), vp(D.ptr(row)), vp(D.ptr(perm)), i64(perm.shape[0]),
                                   vp(D.ptr(out[d])), _sp())
        _lib.check(rc, "b2s_gather")
    return out


def flag_heads(keys):
    t = _t()
    flags = t.empty(keys.shape[0], dtype=t.uint8, device=keys.device)
    _lib.check(_lib.load().b2s_flag_heads(vp(D.ptr(keys)), i64(keys.shape[0]), vp(D.ptr(flags)), _sp()))
    return flags


def flag_not_fill(data, fill_value):
    """keep flags of _prune: bits(data) != bits(fill)  (`equivalent`, _utils.py:448-452)."""
    t = _t()
    flags = t.empty(data.shape[0], dtype=t.uint8, device=data.device)
    buf = _scalar_bytes(fill_value, D.np_dtype(data))
    _lib.check(_lib.load().b2s_flag_not_fill(i32(_esize(data)), vp(D.ptr(data)), i64(data.shape[0]), buf,
                                            vp(D.ptr(flags)), _sp()))
    return flags


def scan_flags(flags):
    """(positions, total)."""
    t = _t()
    pos = t.empty(flags.shape[0], dtype=t.int64, device=flags.device)
    total = ctypes.c_int64(0)
    _lib.check(_lib.load().b2s_scan_flags(vp(D.ptr(flags)), i64(flags.shape[0]), vp(D.ptr(pos)), ctypes.byref(total),
                                         _sp()))
    return pos, int(total.value)


def compact(x, flags, pos, total):
    t = _t()
    out = t.empty(total, dtype=x.dtype, device=x.device)
    _lib.check(_lib.load().b2s_compact(i32(_esize(x)), vp(D.ptr(x)), vp(D.ptr(flags)), vp(D.ptr(pos)),
                                      i64(x.shape[0]), vp(D.ptr(out)), _sp()))
    return out


def compact_rows(x2d, flags, pos, total):
    t = _t()
    if x2d.shape[0] and x2d.stride(1) != 1:
        x2d = x2d.contiguous()
    out = t.empty((x2d.shape[0], total), dtype=x2d.dtype, device=x2d.device)
    if x2d.shape[0] == 0:
        return out
    _lib.check(_lib.load().b2s_compact_rows(i32(_esize(x2d)), i32(x2d.shape[0]), vp(D.ptr(x2d)), i64(x2d.stride(0)),
                                           vp(D.ptr(flags)), vp(D.ptr(pos)), i64(x2d.shape[1]), vp(D.ptr(out)),
                                           i64(max(out.stride(0), 1)), _sp()))
    return out


def segment_sum(data, heads, pos, total):
    """COO._sum_duplicates: sum of every run of equal keys, stored order (_coo/core.py:1350)."""
    t = _t()
    out = t.empty(total, dtype=data.dtype, device=data.device)
    _lib.check(_lib.load().b2s_segment_sum(i32(D.dtype_code(D.np_dtype(data))), vp(D.ptr(data)), vp(D.ptr(heads)),
                                          vp(D.ptr(pos)), i64(data.shape[0]), vp(D.ptr(out)), _sp()))
    return out


def indptr_from_sorted(rows, nrows, idx_dtype=np.int64):
    t = _t()
    out = t.empty(nrows + 1, dtype=D.torch_dtype(idx_dtype), device=rows.device)
    _lib.check(_lib.load().b2s_indptr_from_sorted(i32(_idx_bytes(rows)), vp(D.ptr(rows)), i64(rows.shape[0]),
                                                 i64(nrows), i32(np.dtype(idx_dtype).itemsize), vp(D.ptr(out)),
                                                 _sp()))
    return out


def csr_from_keys(keys, nrows, ncols, idx_dtype=np.int64, want_rows=False, want_indptr=True):
    """Sorted 2-D linear keys -> (rows | None, indices, indptr | None)."""
    t = _t()
    n = keys.shape[0]
    td = D.torch_dtype(idx_dtype)
    indices = t.empty(n, dtype=td, device=keys.device)
    rows = t.empty(n, dtype=td, device=keys.device) if want_rows else None
    indptr = t.empty(nrows + 1, dtype=td, device=keys.device) if want_indptr else None
    _lib.check(_lib.load().b2s_csr_from_keys(vp(D.ptr(keys)), i64(n), i64(nrows), i64(max(ncols, 1)),
                                            i32(np.dtype(idx_dtype).itemsize), vp(D.ptr(rows) if want_rows else 0),
                                            vp(D.ptr(indices)), vp(D.ptr(indptr) if want_indptr else 0), _sp()))
    return rows, indices, indptr


def rows_from_indptr(indptr, nnz, idx_dtype=np.int64):
    """uncompress_dimension (_compressed/convert.py:81-87)."""
    t = _t()
    out = t.empty(nnz, dtype=D.torch_dtype(idx_dtype), device=indptr.device)
    _lib.check(_lib.load().b2s_rows_from_indptr(i32(_idx_bytes(indptr)), vp(D.ptr(indptr)), i64(indptr.shape[0] - 1),
                                               i32(np.dtype(idx_dtype).itemsize), vp(D.ptr(out)), _sp()))
    return out


def full(n, value, dtype):
    """Device buffer of `n` elements set to `value`."""
    t = _t()
    out = t.empty(n, dtype=D.torch_dtype(dtype), device=D.device())
    _lib.check(_lib.load().b2s_fill(i32(out.element_size()), vp(D.ptr(out)), i64(n), _scalar_bytes(value, dtype),
                                   _sp()))
    return out


def iota(n):
    """0..n-1 as int64 (exclusive scan of ones)."""
    pos, _ = scan_flags(full(n, 1, np.uint8))
    return pos


def scatter(data, keys, out):
    """out[keys[i]] = data[i]  (COO.todense)."""
    _lib.check(_lib.load().b2s_scatter(i32(_esize(data)), vp(D.ptr(data)), vp(D.ptr(keys)), i64(keys.shape[0]),
                                      vp(D.ptr(out)), _sp()))
    return out


def cast(x, dtype):
    """Element-wise dtype conversion on the device (C semantics = NumPy astype for the supported dtypes)."""
    t = _t()
    src = D.np_dtype(x)
    dst = np.dtype(dtype)
    if src == dst:
        return x
    if not x.is_contiguous():
        x = x.contiguous()
    out = t.empty(x.shape, dtype=D.torch_dtype(dst), device=x.device)
    _lib.check(_lib.load().b2s_cast(i32(D.cast_code(src)), i32(D.cast_code(dst)), vp(D.ptr(x)), i64(x.numel()),
                                   vp(D.ptr(out)), _sp()))
    return out


def transpose_dense(x):
    """Materialised transpose of a 2-D device tensor (row-major in, row-major out)."""
    t = _t()
    rows, cols = x.shape
    if cols > 1 and x.stride(1) != 1:
        x = x.contiguous()
    out = t.empty((cols, rows), dtype=x.dtype, device=x.device)
    if rows == 0 or cols == 0:
        return out
    _lib.check(_lib.load().b2s_transpose_dense(i32(_esize(x)), vp(D.ptr(x)), i64(rows), i64(cols),
                                              i64(x.stride(0) if rows > 1 else cols), vp(D.ptr(out)), i64(rows),
                                              _sp()))
    return out


def any_nan(x) -> bool:
    dt = D.np_dtype(x)
    if dt.kind != "f":
        return False
    r = ctypes.c_int(0)
    _lib.check(_lib.load().b2s_any_nan(i32(D.dtype_code(dt)), vp(D.ptr(x)), i64(x.numel()), ctypes.byref(r), _sp()))
    return bool(r.value)


def indptr_remap(old_indptr, pos, n, total):
    t = _t()
    out = t.empty_like(old_indptr)
    _lib.check(_lib.load().b2s_indptr_remap(i32(_idx_bytes(old_indptr)), vp(D.ptr(old_indptr)),
                                           i64(old_indptr.shape[0] - 1), vp(D.ptr(pos)), i64(n), i64(total),
                                           vp(D.ptr(out)), _sp()))
    return out


# ------------------------------------------------------------------------------------------------
# K4 SpGEMM
# ------------------------------------------------------------------------------------------------
def spgemm(a_indptr, a_indices, a_data, b_indptr, b_indices, b_data, M, K, n_col, *, sorted_order=False,
           wide=False, prune=False, want_indptr=True, want_rows=False):
    """CSR x CSR -> (indptr | None, indices, rows | None, data, nnz_struct).

    Replaces _dot_csr_csr (_common.py:639-717) / _dot_coo_coo (:907-976); see include/sparse_b200.h.
    """
    t = _t()
    lib = _lib.load()
    dt = D.np_dtype(a_data)
    assert b_data.dtype == a_data.dtype
    idt = a_indptr.dtype
    assert a_indices.dtype == idt and b_indptr.dtype == idt and b_indices.dtype == idt
    plan = ctypes.c_void_p(0)
    n_struct, n_pruned = ctypes.c_int64(0), ctypes.c_int64(0)
    rc = lib.b2s_spgemm_begin(i32(D.dtype_code(dt)), i32(_idx_bytes(a_indptr)), i64(M), i64(K), i64(n_col),
                              vp(D.ptr(a_indptr)), vp(D.ptr(a_indices)), vp(D.ptr(a_data)), vp(D.ptr(b_indptr)),
                              vp(D.ptr(b_indices)), vp(D.ptr(b_data)), i32(1 if sorted_order else 0),
                              i32(1 if wide else 0), ctypes.byref(plan), ctypes.byref(n_struct),
                              ctypes.byref(n_pruned), _sp())
    _lib.check(rc, "b2s_spgemm_begin")
    nnz = int(n_pruned.value) if prune else int(n_struct.value)
    dev = a_data.device
    indices = t.empty(nnz, dtype=t.int64, device=dev)
    data = t.empty(nnz, dtype=a_data.dtype, device=dev)
    indptr = t.empty(M + 1, dtype=t.int64, device=dev) if want_indptr else None
    rows = t.empty(nnz, dtype=t.int64, device=dev) if want_rows else None
    rc = lib.b2s_spgemm_finish(plan, i32(1 if prune else 0), vp(D.ptr(indptr) if want_indptr else 0),
                               vp(D.ptr(indices)), vp(D.ptr(rows) if want_rows else 0), vp(D.ptr(data)))
    _lib.check(rc, "b2s_spgemm_finish")
    return indptr, indices, rows, data, int(n_struct.value)


def spgemm_set_thresholds(t0=64, t1=256):
    _lib.check(_lib.load().b2s_spgemm_set_thresholds(i64(t0), i64(t1)))


# ------------------------------------------------------------------------------------------------
# K3 sparse-output sparse x dense
# ------------------------------------------------------------------------------------------------
def spmm_csr_dense_flagged(a_data, a_indices, a_indptr, b, M, K, N):
    """(out[M,N], flags[M,N]) with _dot_csr_ndarray_sparse arithmetic (_common.py:758-804)."""
    t = _t()
    dt = D.np_dtype(a_data)
    if b.dim() != 2 or (N > 1 and b.stride(1) != 1):
        b = b.contiguous()
    out = t.empty((M, N), dtype=a_data.dtype, device=a_data.device)
    flags = t.empty((M, N), dtype=t.uint8, device=a_data.device)
    ldb = b.stride(0) if K > 1 else max(N, 1)
    _lib.check(_lib.load().b2s_spmm_csr_dense_flagged(
        i32(D.dtype_code(dt)), i32(_idx_bytes(a_indices)), i64(M), i64(K), i64(N), vp(D.ptr(a_data)),
        vp(D.ptr(a_indices)), vp(D.ptr(a_indptr)), vp(D.ptr(b)), i64(max(ldb, N)), vp(D.ptr(out)), vp(D.ptr(flags)),
        _sp()), "b2s_spmm_csr_dense_flagged")
    return out, flags


def dense_to_csr(x, flags=None, mode=0, want_rows=False, want_indptr=True):
    """Dense (M x N) -> (rows | None, cols, data, indptr | None).  mode 0: x != 0, 1: bits != +0."""
    t = _t()
    lib = _lib.load()
    M, N = x.shape
    if not x.is_contiguous():
        x = x.contiguous()
    dt = D.np_dtype(x)
    plan = ctypes.c_void_p(0)
    nnz = ctypes.c_int64(0)
    rc = lib.b2s_dense_to_csr_begin(i32(D.dtype_code(dt)), i64(M), i64(N), vp(D.ptr(x)),
                                    vp(D.ptr(flags) if flags is not None else 0), i32(mode), ctypes.byref(plan),
                                    ctypes.byref(nnz), _sp())
    _lib.check(rc, "b2s_dense_to_csr_begin")
    n = int(nnz.value)
    cols = t.empty(n, dtype=t.int64, device=x.device)
    data = t.empty(n, dtype=x.dtype, device=x.device)
    rows = t.empty(n, dtype=t.int64, device=x.device) if want_rows else None
    indptr = t.empty(M + 1, dtype=t.int64, device=x.device) if want_indptr else None
    rc = lib.b2s_dense_to_csr_finish(plan, vp(D.ptr(rows) if want_rows else 0), vp(D.ptr(cols)), vp(D.ptr(data)),
                                     vp(D.ptr(indptr) if want_indptr else 0))
    _lib.check(rc, "b2s_dense_to_csr_finish")
    return rows, cols, data, indptr


# ------------------------------------------------------------------------------------------------
# K5 elemwise
# ------------------------------------------------------------------------------------------------
def ew_merge_fused(op, keys_a, data_a, Ra, keys_b, data_b, Rb, fill_a, fill_b, out_fill, out_dtype, shape,
                   want_coords=True):
    """Fused COO (x) COO coiteration -> (coords[ndim, nnz] int64, vals[nnz], keys[nnz]); canonical order."""
    t = _t()
    lib = _lib.load()
    dt = D.np_dtype(data_a)
    assert data_b.dtype == data_a.dtype
    cap = int(keys_a.shape[0]) * int(Ra) + int(keys_b.shape[0]) * int(Rb)
    dev = data_a.device
    vals = t.empty(cap, dtype=D.torch_dtype(out_dtype), device=dev)
    keys = t.empty(cap, dtype=t.int64, device=dev)
    nnz = ctypes.c_int64(0)
    rc = lib.b2s_ew_merge_single(
        i32(D.dtype_code(dt)), i32(op), vp(D.ptr(keys_a)), vp(D.ptr(data_a)), i64(keys_a.shape[0]), i64(Ra),
        vp(D.ptr(keys_b)), vp(D.ptr(data_b)), i64(keys_b.shape[0]), i64(Rb), _scalar_bytes(fill_a, dt),
        _scalar_bytes(fill_b, dt), _scalar_bytes(out_fill, out_dtype), i64(cap), vp(D.ptr(vals)), vp(D.ptr(keys)),
        ctypes.byref(nnz), _sp())
    _lib.check(rc, "b2s_ew_merge_single")
    n = int(nnz.value)
    if n != cap:
        # views keep the worst-case buffers alive: give them back when more than a quarter would be wasted
        vals, keys = (vals[:n].clone(), keys[:n].clone()) if 4 * n < 3 * cap else (vals[:n], keys[:n])
    return (unravel(keys, shape, np.int64) if want_coords else None), vals, keys


def ew_map(op, mode, x, scalar, out_fill, out_dtype):
    """f(x, s) (mode 0), f(s, x) (mode 1) or unary f(x) (mode 2) -> (vals, flags)."""
    t = _t()
    dt = D.np_dtype(x)
    n = x.shape[0]
    ovals = t.empty(n, dtype=D.torch_dtype(out_dtype), device=x.device)
    oflags = t.empty(n, dtype=t.uint8, device=x.device)
    rc = _lib.load().b2s_ew_map(i32(D.dtype_code(dt)), i32(op), i32(mode), vp(D.ptr(x)), i64(n),
                               _scalar_bytes(scalar if scalar is not None else 0, dt),
                               _scalar_bytes(out_fill, out_dtype), vp(D.ptr(ovals)), vp(D.ptr(oflags)), _sp())
    _lib.check(rc, "b2s_ew_map")
    return ovals, oflags


def ew_dense(op, swap, keys_a, data_a, Ra, dense, shape, dense_strides, out_fill, out_dtype):
    """COO (x) dense gather -> (keys, vals, flags) with na*Ra slots (_umath.py:606-608)."""
    t = _t()
    dt = D.np_dtype(data_a)
    assert dense.dtype == data_a.dtype
    L = keys_a.shape[0] * Ra
    dev = data_a.device
    okeys = t.empty(L, dtype=t.int64, device=dev)
    ovals = t.empty(L, dtype=D.torch_dtype(out_dtype), device=dev)
    oflags = t.empty(L, dtype=t.uint8, device=dev)
    rc = _lib.load().b2s_ew_dense(i32(D.dtype_code(dt)), i32(op), i32(1 if swap else 0), vp(D.ptr(keys_a)),
                                 vp(D.ptr(data_a)), i64(keys_a.shape[0]), i64(Ra), vp(D.ptr(dense)), i32(len(shape)),
                                 _i64arr(shape), _i64arr(dense_strides), _scalar_bytes(out_fill, out_dtype),
                                 vp(D.ptr(okeys)), vp(D.ptr(ovals)), vp(D.ptr(oflags)), _sp())
    _lib.check(rc, "b2s_ew_dense")
    return okeys, ovals, oflags


def ew_expand(coords, result_shape, is_bcast, src_row):
    """Broadcast expansion over arbitrary axes -> (keys, source index), n * R entries (_umath.py:220-277)."""
    t = _t()
    n = coords.shape[1]
    R = 1
    for d, b in enumerate(is_bcast):
        if b:
            R *= int(result_shape[d])
    L = n * R
    keys = t.empty(L, dtype=t.int64, device=coords.device)
    src = t.empty(L, dtype=t.int64, device=coords.device)
    if coords.shape[0] and coords.stride(1) != 1:
        coords = coords.contiguous()
    rc = _lib.load().b2s_ew_expand(i32(_idx_bytes(coords)), vp(D.ptr(coords)),
                                  i64(coords.stride(0) if coords.shape[0] else 0), i64(n), i32(len(result_shape)),
                                  _i64arr(result_shape), _i32arr(is_bcast), _i32arr(src_row), vp(D.ptr(keys)),
                                  vp(D.ptr(src)), _sp())
    _lib.check(rc, "b2s_ew_expand")
    return keys, src


# ------------------------------------------------------------------------------------------------
# K7 reductions
# ------------------------------------------------------------------------------------------------
def reduce_fused(op, keys, vals, ncols, fill_value, result_fill, kept_shape, want_coords=True):
    """Segmented reduction over runs of key // ncols -> (coords[ndim, g] int64, group ids[g], values[g], n_equal_fill).
    One pass: outputs are allocated for the worst case (one group per entry) and trimmed."""
    t = _t()
    lib = _lib.load()
    dt = D.np_dtype(vals)
    n = int(keys.shape[0])
    dev = vals.device
    gids = t.empty(n, dtype=t.int64, device=dev)
    out = t.empty(n, dtype=vals.dtype, device=dev)
    ng = ctypes.c_int64(0)
    neq = ctypes.c_int64(0)
    rc = lib.b2s_reduce_single(i32(D.dtype_code(dt)), i32(op), vp(D.ptr(keys)), vp(D.ptr(vals)), i64(n), i64(ncols),
                               _scalar_bytes(fill_value, dt), i32(1), _scalar_bytes(result_fill, dt), i64(n),
                               vp(D.ptr(gids)), vp(D.ptr(out)), ctypes.byref(ng), ctypes.byref(neq), _sp())
    _lib.check(rc, "b2s_reduce_single")
    g = int(ng.value)
    if g != n:
        # views keep the worst-case buffers alive: give them back when more than half would be wasted
        gids, out = (gids[:g].clone(), out[:g].clone()) if 2 * g < n else (gids[:g], out[:g])
    coords = unravel(gids, kept_shape, np.int64) if want_coords else None
    return coords, gids, out, int(neq.value)


def reduce_set_form(form: int = 0):
    """Test hook: 0 = choose the reduction kernel by ncols, 1 = single-pass look-back, 2 = count / scan / emit."""
    _lib.check(_lib.load().b2s_reduce_set_form(i32(form)))


# ------------------------------------------------------------------------------------------------
# K8 / K9 fused example paths
# ------------------------------------------------------------------------------------------------
def sddmm(indptr, cols, s_vals, a, bt, M, N, K):
    """out_vals[p] = s_vals[p] * dot(a[i_p], bt[j_p])  (examples/sddmm_example.py:51-52)."""
    t = _t()
    dt = D.np_dtype(s_vals)
    assert a.dtype == s_vals.dtype and bt.dtype == s_vals.dtype and indptr.dtype == cols.dtype
    if K > 1 and a.stride(1) != 1:
        a = a.contiguous()
    if K > 1 and bt.stride(1) != 1:
        bt = bt.contiguous()
    out = t.empty_like(s_vals)
    rc = _lib.load().b2s_sddmm(i32(D.dtype_code(dt)), i32(_idx_bytes(cols)), i64(M), i64(N), i64(K),
                              vp(D.ptr(indptr)), vp(D.ptr(cols)), vp(D.ptr(s_vals)), vp(D.ptr(a)),
                              i64(a.stride(0) if M > 1 else K), vp(D.ptr(bt)), i64(bt.stride(0) if N > 1 else K),
                              vp(D.ptr(out)), _sp())
    _lib.check(rc, "b2s_sddmm")
    return out


def mttkrp(indptr, kk, ll, vals, Dm, Cm, I_, J):
    """out[i, j] = sum_{k,l} B[i,k,l] * D[l,j] * C[k,j]  (examples/mttkrp_example.py:51-52)."""
    t = _t()
    dt = D.np_dtype(vals)
    Dm = Dm.contiguous()
    Cm = Cm.contiguous()
    out = t.empty((I_, J), dtype=vals.dtype, device=vals.device)
    rc = _lib.load().b2s_mttkrp(i32(D.dtype_code(dt)), i32(_idx_bytes(kk)), i64(I_), i64(J), vp(D.ptr(indptr)),
                               vp(D.ptr(kk)), vp(D.ptr(ll)), vp(D.ptr(vals)), vp(D.ptr(Dm)), i64(J), vp(D.ptr(Cm)),
                               i64(J), vp(D.ptr(out)), i64(J), _sp())
    _lib.check(rc, "b2s_mttkrp")
    return out


# ------------------------------------------------------------------------------------------------
# K10 masked sparse product
# ------------------------------------------------------------------------------------------------
def masked_spgemm(s_indptr, s_cols, s_vals, a_indptr, a_indices, a_data, bt_indptr, bt_indices, bt_data, M, N, K):
    """out_vals[p] = s_vals[p] * sum_k a[i_p, k] * bt[j_p, k], ascending k  (`s * (a @ b)` of
    examples/triangles_example.py without the product).  All index arrays share one dtype."""
    t = _t()
    dt_ab = D.np_dtype(a_data)
    assert bt_data.dtype == a_data.dtype
    assert all(x.dtype == s_indptr.dtype for x in (s_cols, a_indptr, a_indices, bt_indptr, bt_indices))
    out = t.empty_like(s_vals)
    rc = _lib.load().b2s_masked_spgemm(i32(D.dtype_code(dt_ab)), i32(D.dtype_code(D.np_dtype(s_vals))),
                                      i32(_idx_bytes(s_indptr)), i64(M), i64(N), i64(K), vp(D.ptr(s_indptr)),
                                      vp(D.ptr(s_cols)), vp(D.ptr(s_vals)), vp(D.ptr(a_indptr)), vp(D.ptr(a_indices)),
                                      vp(D.ptr(a_data)), vp(D.ptr(bt_indptr)), vp(D.ptr(bt_indices)),
                                      vp(D.ptr(bt_data)), vp(D.ptr(out)), _sp())
    _lib.check(rc, "b2s_masked_spgemm")
    return out
