"""Host restatements of the masked sparse product ``s * (a @ b)`` at the stored positions of `s` -- TEST
INFRASTRUCTURE ONLY (the package never imports this module).

* `masked_spgemm_np`: the K10 kernel's contract on CSR arrays with sorted rows, in NumPy: for each mask entry p = (i, j)
  acc = ((+0 + a[i,k1]*bt[j,k1]) + a[i,k2]*bt[j,k2]) + ... over the k stored in both rows in ascending order, products
  and sums rounded in the product dtype (bool: OR of ANDs), then out[p] = s[p] * (out dtype)acc.  It is the CPU mock
  of `Kn.masked_spgemm`.
* `masked_ref_csr`: the same values from an independent route -- the reference's own product kernel restated in C
  (`oracle.dot_csr_csr`, upstream's visiting order, rows stored in any order) gathered at s's positions.  It judges the
  GPU results at sizes the reference cannot run.
"""
from __future__ import annotations

import numpy as np

import oracle


def _mul(x, y):
    with np.errstate(all="ignore"):
        return np.logical_and(x, y) if x.dtype == np.bool_ else x * y


def _add(x, y):
    with np.errstate(all="ignore"):
        return np.logical_or(x, y) if x.dtype == np.bool_ else x + y


def masked_spgemm_np(s_indptr, s_cols, s_vals, a_indptr, a_idx, a_data, bt_indptr, bt_idx, bt_data, M, N, K):
    s_indptr, s_cols, a_indptr, a_idx, bt_indptr, bt_idx = (np.asarray(x, dtype=np.int64) for x in
                                                            (s_indptr, s_cols, a_indptr, a_idx, bt_indptr, bt_idx))
    s_vals, a_data, bt_data = np.asarray(s_vals), np.asarray(a_data), np.asarray(bt_data)
    ta = a_data.dtype
    nnz = len(s_cols)
    rows = np.repeat(np.arange(M, dtype=np.int64), np.diff(s_indptr))
    # every (mask entry, stored k of Bt[j,:]) pair, ascending k inside each entry
    lb = bt_indptr[s_cols + 1] - bt_indptr[s_cols]
    owner = np.repeat(np.arange(nnz, dtype=np.int64), lb)
    start = np.cumsum(lb) - lb
    q = np.repeat(bt_indptr[s_cols], lb) + (np.arange(len(owner), dtype=np.int64) - np.repeat(start, lb))
    k = bt_idx[q]
    # is a[i, k] stored?  keys of A are sorted because its rows are
    a_rows = np.repeat(np.arange(M, dtype=np.int64), np.diff(a_indptr))
    akey = a_rows * max(K, 1) + a_idx
    key = rows[owner] * max(K, 1) + k
    pos = np.searchsorted(akey, key)
    posc = np.minimum(pos, max(len(akey) - 1, 0))
    hit = (pos < len(akey)) & (akey[posc] == key) if len(akey) else np.zeros(len(key), dtype=bool)
    owner, prod = owner[hit], _mul(a_data[pos[hit]], bt_data[q[hit]]).astype(ta)
    # ordered accumulation: the r-th match of every entry is added in round r
    acc = np.zeros(nnz, dtype=ta)
    if len(owner):
        first = np.searchsorted(owner, owner, side="left")
        rank = np.arange(len(owner)) - first
        order = np.argsort(rank, kind="stable")
        bounds = np.searchsorted(rank[order], np.arange(rank.max() + 2))
        for r in range(rank.max() + 1):
            sel = order[bounds[r]:bounds[r + 1]]
            acc[owner[sel]] = _add(acc[owner[sel]], prod[sel])
    return _mul(s_vals, acc.astype(s_vals.dtype)).astype(s_vals.dtype)


def masked_ref_csr(shape, s_indptr, s_cols, s_vals, a_indptr, a_idx, a_data, b_indptr, b_idx, b_data, n_col):
    """s * (a @ b) at s's positions from upstream's CSR @ CSR product (a drives; its rows may be stored in any order).
    s_vals and the result are in the result dtype; a / b values are in their own dtypes."""
    M, N = shape
    c_data, c_idx, c_ptr = oracle.dot_csr_csr((M, n_col), np.asarray(a_data), np.asarray(b_data), a_idx, b_idx,
                                              a_indptr, b_indptr)
    c_rows = np.repeat(np.arange(M, dtype=np.int64), np.diff(c_ptr))
    ckey = c_rows * N + c_idx
    order = np.argsort(ckey, kind="stable")
    ckey, c_data = ckey[order], c_data[order]
    s_rows = np.repeat(np.arange(M, dtype=np.int64), np.diff(np.asarray(s_indptr, dtype=np.int64)))
    skey = s_rows * N + np.asarray(s_cols, dtype=np.int64)
    pos = np.searchsorted(ckey, skey)
    posc = np.minimum(pos, max(len(ckey) - 1, 0))
    found = (pos < len(ckey)) & (ckey[posc] == skey) if len(ckey) else np.zeros(len(skey), dtype=bool)
    acc = np.zeros(len(skey), dtype=c_data.dtype)
    acc[found] = c_data[pos[found]]
    with np.errstate(all="ignore"):
        acc = acc + c_data.dtype.type(0)  # +0 + c: the accumulator of a masked entry is never -0
    s_vals = np.asarray(s_vals)
    return _mul(s_vals, acc.astype(s_vals.dtype)).astype(s_vals.dtype)


def same_bits_nan(x, y):
    """Bitwise equality, NaN payloads aside (the GPU writes the canonical NaN where NumPy keeps an operand's)."""
    x, y = np.asarray(x), np.asarray(y)
    if x.shape != y.shape or x.dtype != y.dtype:
        return False
    if x.dtype.kind != "f":
        return np.array_equal(x, y)
    nx, ny = np.isnan(x), np.isnan(y)
    return np.array_equal(nx, ny) and np.array_equal(x[~nx].view(np.uint8), y[~ny].view(np.uint8))
