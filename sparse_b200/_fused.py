"""Fused SDDMM and MTTKRP: the reference's two example paths as single device kernels.

* sddmm(s, a, b)   == s * (a @ b)                       (examples/sddmm_example.py:51-52)
* mttkrp(B, D, C)  == sparse.sum(B[:, :, :, None] * D[None, None, :, :] * C[None, :, None, :], axis=(1, 2))
                                                        (examples/mttkrp_example.py:51-52)
* masked_matmul(s, a, b) == s * (a @ b) for sparse a, b  (examples/triangles_example.py: sum(a @ a * a))
The unfused expressions also run (through elemwise + reduce); these entry points avoid the dense (a @ b)
intermediate and the nnz x J broadcast products.  For sddmm / mttkrp the floating-point association differs from the
reference's BLAS / reduceat order, so parity is tolerance-based (rtol 1e-5 f32, 1e-12 f64 in the tests);
masked_matmul keeps the reference's order and is bit-exact at the stored positions of `s`.
"""
from __future__ import annotations

import numpy as np

from . import _device as D
from . import _kernels as Kn
from ._coo import COO
from ._dot import _coo_as_csr, _csr_arrays, _dense_dev, _dot_dtype, _is_dense, _narrow_idx
from ._sparse_array import SparseArray
from ._utils import check_zero_fill_value


def _dense_dt(x):
    return x.dtype if isinstance(x, np.ndarray) else D.np_dtype(x)


def sddmm(s, a, b, *, b_transposed=False):
    """Sampled dense-dense matrix product: ``s * (a @ b)`` for sparse 2-D ``s`` and dense ``a`` (M,K), ``b`` (K,N).
    With ``b_transposed=True`` `b` is given as b^T (N,K), the layout the kernel gathers from."""
    from ._gcxs import GCXS

    if not isinstance(s, SparseArray) or s.ndim != 2:
        raise TypeError("sddmm: `s` must be a 2-D sparse_b200 array")
    check_zero_fill_value(s)
    M, N = s.shape
    if b_transposed:
        bN, bK = int(b.shape[0]), int(b.shape[1])
    else:
        bK, bN = int(b.shape[0]), int(b.shape[1])
    if a.ndim != 2 or b.ndim != 2 or a.shape[0] != M or bN != N or a.shape[1] != bK:
        raise ValueError(f"sddmm: shape mismatch s{s.shape}, a{tuple(a.shape)}, b{tuple(b.shape)}")
    K = int(a.shape[1])
    T = np.result_type(s.dtype, _dense_dt(a), _dense_dt(b))
    if T not in (np.dtype("float32"), np.dtype("float64")):
        raise TypeError(f"sddmm: dtype {T} is outside the CUDA dtype matrix (float32, float64)")
    was_gcxs = isinstance(s, GCXS)
    c = s.tocoo() if was_gcxs else s
    vals, cols, indptr = _coo_as_csr(c, T)
    ad = _dense_dev(a, T)
    bt = _dense_dev(b, T) if b_transposed else Kn.transpose_dense(_dense_dev(b, T))  # (N, K): contiguous gathers
    out = Kn.sddmm(indptr, cols, vals, ad, bt, M, N, K)
    fill = T.type(0)
    if isinstance(a, np.ndarray) and isinstance(b, np.ndarray) and M and N and K:
        # the unfused expression's fill value is `0 * (a @ b)[0, 0]` (_umath.py:520-527: the first element of
        # func(fill, ndarray)), i.e. -0.0 when that corner is negative -- and the prune test below is by bit pattern,
        # so the sign decides WHICH zeros stay stored.  K multiply-adds on the host; device operands keep +0.0
        # (no read-back on the asynchronous path)
        with np.errstate(all="ignore"):
            corner = np.dot(a[0].astype(T, copy=False), (b[0] if b_transposed else b[:, 0]).astype(T, copy=False))
            if np.isfinite(corner):
                fill = T.type(T.type(0) * (corner + T.type(0)))  # a sum that starts at +0.0 is never -0.0
    res = COO._from_device(c._coords, out, s.shape, fill, keys=c.sorted_keys())
    res._canonicalise(check_sort=False, sum_dups=False, prune=True)  # s * dense drops exact zeros (_umath.py:627-633)
    return res.asformat("gcxs", compressed_axes=s.compressed_axes) if was_gcxs else res


def mttkrp(B, Dm, Cm):
    """Matricised tensor times Khatri-Rao product: out[i, j] = sum_{k,l} B[i,k,l] * D[l,j] * C[k,j]."""
    from ._gcxs import GCXS

    if not isinstance(B, SparseArray) or B.ndim != 3:
        raise TypeError("mttkrp: `B` must be a 3-D sparse_b200 array")
    check_zero_fill_value(B)
    I_, K_, L_ = B.shape
    if Dm.ndim != 2 or Cm.ndim != 2 or Dm.shape[0] != L_ or Cm.shape[0] != K_ or Dm.shape[1] != Cm.shape[1]:
        raise ValueError(f"mttkrp: shape mismatch B{B.shape}, D{tuple(Dm.shape)}, C{tuple(Cm.shape)}")
    J = int(Dm.shape[1])
    T = np.result_type(B.dtype, _dense_dt(Dm), _dense_dt(Cm))
    if T not in (np.dtype("float32"), np.dtype("float64")):
        raise TypeError(f"mttkrp: dtype {T} is outside the CUDA dtype matrix (float32, float64)")
    was_gcxs = isinstance(B, GCXS)
    c = B.tocoo() if was_gcxs else B
    coords, data = c._dev()
    c.sorted_keys()
    lead = coords[0].contiguous()
    indptr = Kn.indptr_from_sorted(lead, I_, D.np_dtype(coords))
    kk, ll, indptr = _narrow_idx(coords[1].contiguous(), coords[2].contiguous(), indptr, limit=max(K_, L_, c.nnz))
    out = Kn.mttkrp(indptr, kk, ll, Kn.cast(data, T), _dense_dev(Dm, T), _dense_dev(Cm, T), I_, J)
    rows, cols, vals, _ = Kn.dense_to_csr(out, mode=1, want_rows=True, want_indptr=False)
    t = D.torch()
    res = COO._from_device(t.stack([rows, cols]), vals, (I_, J), T.type(0))
    return GCXS.from_coo(res) if was_gcxs else res


_F32, _F64, _I64, _BOOL = np.dtype("float32"), np.dtype("float64"), np.dtype("int64"), np.dtype("bool")


def _masked_types(t_ab, t_out):
    """(accumulator dtype, kernel output dtype, wrap) of K10 for the product dtype `t_ab` and the result dtype `t_out`.
    Integer products are computed in int64 and cast back: sums and products that wrap modulo 2**64 wrap to the same
    bits in every narrower integer type (the wide-compute path of `_dot`'s `_WIDE_FOR`).  `wrap`: an integer product
    narrower than int64 (or unsigned) under a floating-point result -- the kernel then writes the int64 sums alone, and
    the host casts them to `t_ab` (where they wrap as upstream's) and multiplies by `s` in `t_out`."""
    if t_ab in (_F32, _F64) and t_out in (_F32, _F64):
        return t_ab, t_out, False
    if t_ab == _BOOL and t_out in (_BOOL, _F32, _F64):
        return _BOOL, t_out, False
    if t_ab == _BOOL and t_out.kind in "iu":
        return _BOOL, _I64, False
    if t_ab.kind in "iu" and t_out.kind in "iu":
        return _I64, _I64, False
    if t_ab == _I64 and t_out == _F64:
        return _I64, _F64, False
    if t_ab.kind in "iu" and t_out in (_F32, _F64):
        return _I64, _I64, True
    raise TypeError(f"masked_matmul: product dtype {t_ab} with result dtype {t_out} is outside the CUDA dtype matrix")


def masked_matmul(s, a, b):
    """Masked sparse product ``s * (a @ b)`` for sparse 2-D ``s``, ``a``, ``b`` (COO / GCXS, zero fill values), without
    forming ``a @ b``: work and memory grow with the mask and the rows it touches, not with the products of ``a @ b``.
    Dense ``a`` and ``b`` go to :func:`sddmm`.

    For every stored position p = (i, j) of `s`: ``out[p] = s[p] * acc(i, j)`` in the result dtype
    ``np.result_type(s.dtype, a @ b's dtype)`` (both sides cast to it first), where
    ``acc(i, j) = ((+0 + a[i,k1]*b[k1,j]) + a[i,k2]*b[k2,j]) + ...`` over the matching k in the reference's visiting
    order (ascending k for sorted rows), each product rounded to the dtype of ``a @ b``, no fused multiply-add.  Values
    bitwise equal to +0 are dropped.  The result's class and compressed axes are those of the unfused expression.

    The result equals the reference's ``s * (a @ b)`` at the stored positions of `s`.  The unfused expression may also
    store entries of ``a @ b`` outside `s` where ``0 * v`` is not +0 (a -0.0 from a negative v, a NaN from an infinite
    or NaN v); they are not computed here.  Without negative or non-finite entries of ``a @ b`` outside `s` (e.g. 0/1
    graph adjacency) the two are equal outright."""
    from ._dot import matmul
    from ._gcxs import GCXS

    if _is_dense(a) and _is_dense(b):
        return sddmm(s, a, b)
    if not all(isinstance(x, (COO, GCXS)) for x in (s, a, b)):
        raise TypeError("masked_matmul: expected sparse s, a, b (COO / GCXS), or a sparse s with dense a, b (sddmm); "
                        f"got {type(s).__name__}, {type(a).__name__}, {type(b).__name__}")
    if any(x.dtype.kind == "c" for x in (s, a, b)):
        raise TypeError("masked_matmul: complex operands are not supported")
    if s.ndim != 2 or a.ndim != 2 or b.ndim != 2:
        raise ValueError(f"masked_matmul: 2-D operands expected, got s{s.shape}, a{a.shape}, b{b.shape}")
    check_zero_fill_value(s, a, b)
    M, N = s.shape
    K = a.shape[1]
    if a.shape[0] != M or tuple(b.shape) != (K, N):
        raise ValueError(f"masked_matmul: shape mismatch s{s.shape}, a{a.shape}, b{b.shape}")

    # format and dtype of the reference's `a @ b` (tensordot / _dot): an empty COO when an axis has length 0, else GCXS
    # compressed like `a` (a COO `a` gets from_coo's default, the shorter axis) as soon as one operand is GCXS
    if M == 0 or N == 0 or K == 0:
        t_ab, prod_ca = np.result_type(a.dtype, b.dtype), None
    else:
        t_ab = _dot_dtype(a.dtype, b.dtype)
        prod_ca = None
        if isinstance(a, GCXS) or isinstance(b, GCXS):
            prod_ca = a.compressed_axes if isinstance(a, GCXS) else (int(np.argmin(a.shape)),)
    t_out = np.result_type(s.dtype, t_ab)
    t_acc, t_k, wrap = _masked_types(t_ab, t_out)

    sc = s.tocoo() if isinstance(s, GCXS) else s
    if sc.nnz == 0 or M == 0 or N == 0:
        coords, data = sc._dev()
        res = COO._from_device(coords, Kn.cast(data, t_out), s.shape, t_out.type(0))
    else:
        sv, scols, sptr = _coo_as_csr(sc, t_k)
        if wrap:
            sv = Kn.full(sc.nnz, 1, _I64)  # unit mask: the kernel returns the int64 sums themselves
        # The reference sums in the stored order of the row that drives its product: a's row (CSR product) or b's column
        # (CSC product).  That is ascending k unless the driver is a GCXS stored with unsorted rows (e.g. the result of
        # an earlier GCXS @ GCXS); for a floating-point sum the exact route is then the reference's product itself,
        # gathered at s's positions by the same kernel with an identity for b: +0 + c[i,j] * 1 == c[i,j].
        driver = a if prod_ca == (0,) else b if prod_ca == (1,) else None
        unsorted = (isinstance(driver, GCXS) and driver.compressed_axes == prod_ca and t_acc.kind == "f"
                    and driver.nnz > 0 and not driver._rows_sorted())
        if unsorted:
            c = matmul(a, b)
            ad, ai, ap = _coo_as_csr(c.tocoo() if isinstance(c, GCXS) else c, t_acc)
            bi, bp = Kn.iota(N), Kn.iota(N + 1)
            bd = Kn.full(N, 1, t_acc)
        else:
            # a CSR `a` / CSC `b` with sorted rows already holds the arrays the kernel reads (A by row, Bt = b by column)
            if isinstance(a, GCXS) and a.compressed_axes == (0,) and a._rows_sorted():
                ad, ai, ap = _csr_arrays(a, t_acc)
            else:
                ad, ai, ap = _coo_as_csr(a.tocoo() if isinstance(a, GCXS) else a, t_acc)
            if isinstance(b, GCXS) and b.compressed_axes == (1,) and b._rows_sorted():
                bd, bi, bp = _csr_arrays(b, t_acc)
            else:
                bd, bi, bp = _coo_as_csr(b.tocoo() if isinstance(b, GCXS) else b, t_acc, by_col=True)
        idx = [sptr, scols, ap, ai, bp, bi]
        t = D.torch()
        if any(x.dtype != idx[0].dtype for x in idx):
            idx = [x if x.dtype == t.int64 else Kn.cast(x, np.int64) for x in idx]
        sptr, scols, ap, ai, bp, bi = idx
        out = Kn.masked_spgemm(sptr, scols, sv, ap, ai, ad, bp, bi, bd, M, N, K)
        if wrap:
            from ._elemwise import dense_binary

            out = dense_binary(np.multiply, Kn.cast(sc._data_dev(), t_out), Kn.cast(Kn.cast(out, t_ab), t_out))
        res = COO._from_device(sc._coords, Kn.cast(out, t_out), s.shape, t_out.type(0), keys=sc.sorted_keys())
        res._canonicalise(check_sort=False, sum_dups=False, prune=True)  # drop values bitwise equal to +0
    if isinstance(s, GCXS) and prod_ca is not None:
        # the element-wise result format: GCXS, with s's compressed axes when the product has the same ones
        return res.asformat(GCXS, **({"compressed_axes": s.compressed_axes} if s.compressed_axes == prod_ca else {}))
    return res
