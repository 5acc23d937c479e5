#!/usr/bin/env python
"""Differential fuzzing of the host layer against the REFERENCE itself (authoring container only).

    python tools/fuzz_vs_reference.py [--cases 3000] [--seed 0] [--family all|join,methods,nary,where,special,fused,io,helpers,einsum,scipy,dot,elemwise,reduce,formats,protocol]
                                      [--only CASE] [-v]

Both packages live in one process: the reference is imported from oracle/_ref (oracle/make_ref.sh: the unmodified
upstream package, numba kernels), this package runs on the NumPy mock of the kernel layer (tests/_mock_kernels.py) when
there is no GPU -- then what is fuzzed is everything ABOVE the C ABI (on a GPU box the CUDA kernels run instead): axis bookkeeping, broadcasting, dtype promotion,
fill values, result formats, error classes.  The kernels are compared with the oracle / golden vectors on the GPU
(tests/, -m gpu).  Random shapes (0-4 dims, zero-length axes included), densities, dtypes, fill values, formats,
operators; every result is compared field by field: class, shape, dtype, fill value, and the stored entries EXACTLY
(COO: coords + data; GCXS: compressed axes, indptr, indices -- including the reference's unsorted column order after a
CSR x CSR product -- and data).  Inputs are small integers stored in the drawn dtype, so every sum is exact in any order.
An exception on one side must be the same class on the other.  Every mismatch prints a reproducer line
(`--family F --seed S --only CASE -v` re-runs it).

Counted but not reported (each with the reason next to the code that recognises it): crashes INSIDE the reference on
degenerate input, reference results that NumPy contradicts while this package agrees with NumPy, garbage entries from
the uninitialised tail of `_dot_csc_ndarray_sparse`.  Left out of the
draws because the answer is a documented `TypeError` here (DESIGN s4): ops outside the CUDA op set (hypot, arctan2,
copysign), integer power in narrow dtypes, float16 results.

Nothing here is imported by the product, the tests, or bench.py.
"""
from __future__ import annotations

import argparse
import os
import sys
import traceback
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)

import sparse as R  # noqa: E402  (the reference)

import torch  # noqa: E402

if not torch.cuda.is_available():  # authoring container: the NumPy mock of the kernel layer; on a GPU box
    import _mock_kernels  # noqa: E402   the real CUDA kernels are fuzzed

    _mock_kernels.install()
import sparse_b200 as S  # noqa: E402

assert "oracle/_ref" in R.__file__, R.__file__

FLOATS = ["float64", "float32"]
INTS = ["int64", "int32", "int16", "int8", "uint8", "uint32"]
DTYPES = FLOATS * 3 + INTS + ["bool"]


def eq_scalar(a, b):
    a, b = np.asarray(a), np.asarray(b)
    if a.dtype != b.dtype:
        return False
    return bool(np.array_equal(a, b, equal_nan=a.dtype.kind in "fc"))


def arr_eq(a, b):
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape:
        return False
    if a.dtype.kind in "fc" or b.dtype.kind in "fc":
        return bool(np.array_equal(a, b, equal_nan=True))
    return bool(np.array_equal(a, b))


def compare(got, want, exact_layout=True):
    """None when equal, else a description."""
    if isinstance(want, R.COO):
        if not isinstance(got, S.COO):
            return f"class {type(got).__name__} != COO"
        if tuple(got.shape) != tuple(want.shape):
            return f"shape {got.shape} != {want.shape}"
        if got.dtype != want.dtype:
            return f"dtype {got.dtype} != {want.dtype}"
        if not eq_scalar(got.fill_value, want.fill_value):
            return f"fill {got.fill_value!r} ({np.asarray(got.fill_value).dtype}) != {want.fill_value!r} ({np.asarray(want.fill_value).dtype})"
        if exact_layout:
            if not arr_eq(np.asarray(got.coords), want.coords):
                if arr_eq(got.todense(), want.todense()):
                    return f"coords differ (dense equal): nnz {got.nnz} vs {want.nnz}"
                return "coords differ and dense differs"
            if not arr_eq(np.asarray(got.data), want.data):
                return "data differ"
        elif not arr_eq(got.todense(), want.todense()):
            return "dense differs"
        return None
    if isinstance(want, R.GCXS):
        if not isinstance(got, S.GCXS):
            return f"class {type(got).__name__} != GCXS"
        if tuple(got.shape) != tuple(want.shape):
            return f"shape {got.shape} != {want.shape}"
        if got.dtype != want.dtype:
            return f"dtype {got.dtype} != {want.dtype}"
        if not eq_scalar(got.fill_value, want.fill_value):
            return f"fill {got.fill_value!r} != {want.fill_value!r}"
        ca_g = tuple(got.compressed_axes) if got.compressed_axes is not None else None
        ca_w = tuple(want.compressed_axes) if want.compressed_axes is not None else None
        if ca_g != ca_w:
            return f"compressed_axes {ca_g} != {ca_w}"
        if exact_layout:
            if not arr_eq(np.asarray(got.indptr), np.asarray(want.indptr)):
                return "indptr differ" + (" (dense equal)" if arr_eq(got.todense(), want.todense()) else "")
            if not arr_eq(np.asarray(got.indices), want.indices):
                return "indices differ" + (" (dense equal)" if arr_eq(got.todense(), want.todense()) else "")
            if not arr_eq(np.asarray(got.data), want.data):
                return "data differ"
        elif not arr_eq(got.todense(), want.todense()):
            return "dense differs"
        return None
    if isinstance(want, R.DOK):
        if not isinstance(got, S.DOK):
            return f"class {type(got).__name__} != DOK"
        return None if arr_eq(got.todense(), want.todense()) else "dense differs"
    if isinstance(got, S.SparseArray):
        return f"class {type(got).__name__} != {type(want).__name__}"
    g, w = np.asarray(got), np.asarray(want)
    if g.shape != w.shape:
        return f"dense shape {g.shape} != {w.shape}"
    if g.dtype != w.dtype:
        return f"dense dtype {g.dtype} != {w.dtype}"
    if not arr_eq(g, w):
        return "dense values differ"
    if isinstance(want, np.ndarray) != isinstance(got, np.ndarray) and not (np.isscalar(want) or np.isscalar(got)):
        return f"container {type(got).__name__} != {type(want).__name__}"
    return None


MAX_EXTENT = [6]  # --max-extent: exclusive upper bound of the drawn axis lengths (elemwise / reduce / formats ...)


def draw_shape(rng, lo=0, hi=4, zero_ok=True):
    nd = int(rng.integers(lo, hi + 1))
    return tuple(int(rng.integers(0 if (zero_ok and rng.random() < 0.07) else 1, MAX_EXTENT[0])) for _ in range(nd))


def draw_dense(rng, shape, dtype, density=None, fill=0):
    density = rng.choice([0.0, 0.15, 0.5, 1.0]) if density is None else density
    dt = np.dtype(dtype)
    if dt.kind == "b":
        vals = rng.random(shape) < 0.5
        d = np.full(shape, bool(fill), dtype=dt)
    else:
        lo = 0 if dt.kind == "u" else -4
        vals = rng.integers(lo, 5, size=shape).astype(dt)
        d = np.full(shape, fill, dtype=dt)
    mask = rng.random(shape) < density
    d[mask] = vals[mask]
    return d


def both(d, fmt, fill=0, rng=None):
    """The same array in both packages (fmt: coo | gcxs | dense)."""
    if fmt == "dense":
        return d, d
    fv = np.asarray(fill, dtype=d.dtype)[()]
    r = R.COO.from_numpy(d, fill_value=fv)
    s = S.COO.from_numpy(d, fill_value=fv)
    if fmt == "gcxs":
        kw = {}
        if d.ndim >= 2 and rng is not None and rng.random() < 0.5:
            k = int(rng.integers(1, d.ndim))
            kw["compressed_axes"] = tuple(sorted(int(x) for x in rng.choice(d.ndim, size=k, replace=False)))
        r = r.asformat("gcxs", **kw)
        s = s.asformat("gcxs", **kw)
    return s, r


def run_pair(f_s, f_r):
    """Run both sides; returns (got, want, err_s, err_r)."""
    got = want = es = er = None
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        try:
            want = f_r()
        except Exception as e:  # noqa: BLE001
            er = e
        try:
            got = f_s()
        except Exception as e:  # noqa: BLE001
            es = e
    return got, want, es, er


def ref_crash(er):
    """Crashes INSIDE the reference on degenerate input -- a zero-length contraction (ZeroDivisionError), all axes of a
    GCXS array given as a permuted tuple (min() of an empty list), the fill value's contribution computed in a narrow
    dtype (OverflowError).  A result here (NumPy's) is not a parity failure."""
    return (isinstance(er, ZeroDivisionError) or "min() iterable argument is empty" in str(er)
            or "invalid entry in coordinates array" in str(er)  # garbage indices from the uninitialised tail (s4)
            or "has no attribute '_compressed_axes'" in str(er)  # a GCXS object upstream left half-built
            or (isinstance(er, OverflowError) and "out of bounds for" in str(er)))


def _has_duplicate_indices(g):
    ip, ix = np.asarray(g.indptr).astype(np.int64), np.asarray(g.indices)
    return any(len(np.unique(ix[ip[r]:ip[r + 1]])) < ip[r + 1] - ip[r] for r in range(len(ip) - 1))


class Stats:
    def __init__(self, verbose):
        self.n = self.bad = self.errs_both = self.ref_crashes = self.ref_wrong = self.unmockable = 0
        self.kinds = {}
        self.verbose = verbose

    def report(self, family, desc, msg):
        self.bad += 1
        key = (family, msg.split(":")[0][:60])
        self.kinds[key] = self.kinds.get(key, 0) + 1
        if self.kinds[key] <= 3 or self.verbose:
            print(f"MISMATCH [{family}] {desc}\n    -> {msg}", flush=True)

    def check(self, family, desc, f_s, f_r, exact_layout=True, truth=None):
        """`truth`: NumPy's dense answer where one exists -- a reference result that disagrees with it while this
        package agrees (the uninitialised tail `_dot_csc_ndarray_sparse` reads, DESIGN s4) is counted, not reported."""
        self.n += 1
        got, want, es, er = run_pair(f_s, f_r)
        if truth is not None and es is None and er is None:
            try:
                t = truth()
                dense = lambda v: v.todense() if hasattr(v, "todense") else np.asarray(v)  # noqa: E731
                if not arr_eq(dense(want), t) and arr_eq(dense(got), t):
                    self.ref_wrong += 1
                    return
            except Exception:  # noqa: BLE001
                pass
        if er is not None or es is not None:
            if er is not None and es is not None:
                self.errs_both += 1
                if type(es).__name__ != type(er).__name__ and not isinstance(es, type(er)):
                    self.report(family, desc, f"error class: {type(es).__name__}({es}) != {type(er).__name__}({er})")
                return
            if es is not None and "no CUDA device visible" in str(es):
                self.unmockable += 1  # a path without a mock (none left: the host-buffer product has one now)
                return
            if er is not None and ref_crash(er):
                self.ref_crashes += 1
                return
            if er is not None:
                self.report(family, desc, f"reference raised {type(er).__name__}({er}); here: result")
            else:
                tb = traceback.format_exception(type(es), es, es.__traceback__)[-3:]
                self.report(family, desc, f"here raised {type(es).__name__}({es}); reference: result\n      " +
                            "      ".join(tb))
            return
        msg = compare(got, want, exact_layout)
        if msg and isinstance(want, R.GCXS) and want.ndim >= 2 and _has_duplicate_indices(want):
            self.ref_wrong += 1  # entries of the uninitialised tail (same column twice in one row, denormal values)
            return
        if msg:
            self.report(family, desc, msg)


# ------------------------------------------------------------------------------------------------------------ families
def fam_dot(rng, st, i):
    kind = rng.choice(["tensordot", "matmul", "dot"])
    dt_a, dt_b = rng.choice(DTYPES[:-1]), rng.choice(DTYPES[:-1])
    fa, fb = rng.choice(["coo", "gcxs", "dense"]), rng.choice(["coo", "gcxs", "dense"])
    if fa == "dense" and fb == "dense":
        fa = "coo"
    if kind == "tensordot":
        nd_a, nd_b = int(rng.integers(1, 5)), int(rng.integers(1, 5))
        k = int(rng.integers(0, min(nd_a, nd_b) + 1))
        ax_a = [int(x) for x in rng.choice(nd_a, size=k, replace=False)]
        ax_b = [int(x) for x in rng.choice(nd_b, size=k, replace=False)]
        sa = [int(rng.integers(1, max(5, MAX_EXTENT[0] - 1))) for _ in range(nd_a)]
        sb = [int(rng.integers(1, max(5, MAX_EXTENT[0] - 1))) for _ in range(nd_b)]
        for x, y in zip(ax_a, ax_b):
            sb[y] = sa[x]
        if rng.random() < 0.05 and k:
            sb[ax_b[0]] += 1  # shape mismatch -> error parity
        if rng.random() < 0.06:
            sa[int(rng.integers(nd_a))] = 0
            for x, y in zip(ax_a, ax_b):
                sb[y] = sa[x]
        form = rng.random()
        if form < 0.25 and k and ax_a == list(range(nd_a - k, nd_a)) and ax_b == list(range(k)):
            axes = k
        elif form < 0.4 and k == 1:
            axes = (ax_a[0] - (nd_a if rng.random() < 0.5 else 0), ax_b[0])
        else:
            axes = (ax_a, ax_b)
        rt_name = rng.choice(["none", "none", "coo", "gcxs", "dense"])
    else:
        K = int(rng.integers(1, max(5, MAX_EXTENT[0] - 1)))
        if kind == "matmul":
            batch = draw_shape(rng, 0, 2, zero_ok=False)
            ba = tuple(1 if rng.random() < 0.3 else b for b in batch)[int(rng.integers(0, len(batch) + 1)):]
            bb = tuple(1 if rng.random() < 0.3 else b for b in batch)[int(rng.integers(0, len(batch) + 1)):]
            sa = list(ba) + ([int(rng.integers(1, max(5, MAX_EXTENT[0] - 1)))] if rng.random() < 0.85 or ba else []) + [K]
            sb = list(bb) + [K] + ([int(rng.integers(1, max(5, MAX_EXTENT[0] - 1)))] if rng.random() < 0.85 or bb else [])
        else:
            sa = list(draw_shape(rng, 0, 2, zero_ok=False)) + [K]
            sb = list(draw_shape(rng, 0, 1, zero_ok=False)) + [K] + ([int(rng.integers(1, max(5, MAX_EXTENT[0] - 1)))] if rng.random() < 0.8 else [])
            if len(sb) == 1:
                pass
        axes, rt_name = None, "none"
    da = draw_dense(rng, tuple(sa), dt_a)
    db = draw_dense(rng, tuple(sb), dt_b)
    a_s, a_r = both(da, fa, rng=rng)
    b_s, b_r = both(db, fb, rng=rng)
    rts_s = {"none": None, "coo": S.COO, "gcxs": S.GCXS, "dense": np.ndarray}
    rts_r = {"none": None, "coo": R.COO, "gcxs": R.GCXS, "dense": np.ndarray}
    ca = lambda x: getattr(x, "compressed_axes", None)  # noqa: E731
    desc = (f"#{i} {kind} a={fa}{tuple(sa)}:{dt_a} ca={ca(a_r)} b={fb}{tuple(sb)}:{dt_b} ca={ca(b_r)} axes={axes} "
            f"rt={rt_name}")
    if kind == "tensordot" and rt_name == "none" and rng.random() < 0.3:
        st.check("dot", desc + " via=numpy", lambda: np.tensordot(a_s, b_s, axes), lambda: np.tensordot(a_r, b_r, axes),
                 truth=lambda: np.tensordot(da, db, axes))
    elif kind == "tensordot":
        st.check("dot", desc, lambda: S.tensordot(a_s, b_s, axes, return_type=rts_s[rt_name]),
                 lambda: R.tensordot(a_r, b_r, axes, return_type=rts_r[rt_name]),
                 truth=lambda: np.tensordot(da, db, axes))
    elif kind == "matmul":
        # the module function, the operator (also with the ndarray on the left: __rmatmul__ / __array_ufunc__) and
        # NumPy's own entry point (__array_function__)
        via = rng.choice(["func", "operator", "numpy"])
        call = {"func": lambda m, x, y: m.matmul(x, y), "operator": lambda m, x, y: x @ y,
                "numpy": lambda m, x, y: np.matmul(x, y)}[via]
        st.check("dot", desc + f" via={via}", lambda: call(S, a_s, b_s), lambda: call(R, a_r, b_r),
                 truth=lambda: np.matmul(da, db))
    else:
        via = rng.choice(["func", "method", "numpy"])
        if via == "method" and fa == "dense":
            via = "func"
        call = {"func": lambda m, x, y: m.dot(x, y), "method": lambda m, x, y: x.dot(y),
                "numpy": lambda m, x, y: np.dot(x, y)}[via]
        st.check("dot", desc + f" via={via}", lambda: call(S, a_s, b_s), lambda: call(R, a_r, b_r),
                 truth=lambda: np.dot(da, db))


BINARY = ["add", "subtract", "multiply", "maximum", "minimum", "greater", "less", "greater_equal", "less_equal",
          "equal", "not_equal", "true_divide", "floor_divide", "power", "logical_and", "logical_or", "logical_xor",
          "bitwise_and", "bitwise_or", "bitwise_xor", "remainder", "fmax", "fmin"]  # hypot, arctan2, copysign: outside the CUDA op set (TypeError by design)
UNARY = ["negative", "abs", "sign", "square", "sqrt", "sin", "expm1", "log1p", "tanh", "isnan", "isfinite", "floor",
         "ceil", "rint", "logical_not", "exp", "cos", "positive", "conj", "invert", "signbit", "trunc", "deg2rad"]


F16_FROM_8BIT = {"sqrt", "sin", "expm1", "log1p", "tanh", "exp", "cos", "deg2rad", "floor", "ceil", "rint", "trunc"}


def fam_elemwise(rng, st, i):
    mode = rng.choice(["binary", "binary", "binary", "unary", "scalar", "nary"])
    base = draw_shape(rng, 0, 4)
    dt_a = rng.choice(DTYPES)
    fill_a = rng.choice([0, 0, 0, 1, 2]) if dt_a != "bool" else rng.choice([0, 0, 1])
    fa = rng.choice(["coo", "coo", "gcxs"])
    da = draw_dense(rng, base, dt_a, fill=fill_a)
    a_s, a_r = both(da, fa, fill=fill_a, rng=rng)
    if mode == "unary":
        name = rng.choice(UNARY)
        if np.dtype(dt_a).itemsize == 1 and name in F16_FROM_8BIT:
            name = "negative" if dt_a != "bool" else "logical_not"  # float16 loops: outside the CUDA dtype matrix
        f = getattr(np, name)
        st.check("elemwise", f"#{i} np.{name}({fa}{base}:{dt_a} fill={fill_a})", lambda: f(a_s), lambda: f(a_r))
        return
    if mode == "scalar":
        name = rng.choice(BINARY)
        f = getattr(np, name)
        if name == "power" and (np.dtype(dt_a).itemsize < 4 or dt_a == "uint32"):
            name, f = "multiply", np.multiply  # integer power in a narrow / unsigned type: documented TypeError
        sc = rng.choice([0, 1, 2, -1, 2.5, True, np.float32(3), np.int8(2), np.float64("nan")])
        if rng.random() < 0.3:  # a 0-D ndarray operand (strongly typed, unlike a Python scalar)
            sc = np.array(rng.integers(0, 4)).astype(rng.choice(["float64", "float32", "int64", "int8", "bool"]))
        kw = {}
        if rng.random() < 0.2 and name in ("add", "multiply", "subtract", "maximum", "minimum", "true_divide"):
            kw["dtype"] = rng.choice(["float64", "float32"])  # selects the loop: operands are cast first
        left = rng.random() < 0.5
        st.check("elemwise", f"#{i} np.{name}({'scalar,' if left else ''}{fa}{base}:{dt_a} fill={fill_a}"
                             f"{'' if left else ',scalar'}, {kw}) scalar={sc!r}",
                 (lambda: f(sc, a_s, **kw)) if left else (lambda: f(a_s, sc, **kw)),
                 (lambda: f(sc, a_r, **kw)) if left else (lambda: f(a_r, sc, **kw)))
        return
    # second operand: a broadcast-compatible shape
    other = tuple(s if rng.random() < 0.65 else 1 for s in base)
    other = other[int(rng.integers(0, len(other) + 1)):]
    if rng.random() < 0.2:
        other = tuple(int(rng.integers(1, 4)) for _ in range(int(rng.integers(0, 2)))) + other
    if rng.random() < 0.04 and other:
        other = other[:-1] + (other[-1] + 1,)  # incompatible -> error parity
    dt_b = rng.choice(DTYPES)
    fill_b = rng.choice([0, 0, 0, 1, 3]) if dt_b != "bool" else rng.choice([0, 0, 1])
    fb = rng.choice(["coo", "coo", "gcxs", "dense"])
    db = draw_dense(rng, other, dt_b, fill=fill_b)
    b_s, b_r = both(db, fb, fill=fill_b, rng=rng)
    if mode == "nary":
        dc = draw_dense(rng, base, rng.choice(FLOATS + ["int64"]))
        c_s, c_r = both(dc, "coo")
        which = rng.choice(["where", "fma", "clip"])
        if which == "where":
            st.check("elemwise", f"#{i} where(a{base}:{dt_a}!=0, b{other}:{dt_b} {fb}, c)",
                     lambda: S.where(a_s != 0, b_s, c_s), lambda: R.where(a_r != 0, b_r, c_r))
        elif which == "fma":
            st.check("elemwise", f"#{i} elemwise(lambda x,y,z: x*y+z) a{base}:{dt_a} f={fill_a} b{other}:{dt_b} {fb} f={fill_b}",
                     lambda: S.elemwise(lambda x, y, z: x * y + z, a_s, b_s, c_s),
                     lambda: R.elemwise(lambda x, y, z: x * y + z, a_r, b_r, c_r))
        else:
            st.check("elemwise", f"#{i} clip a{base}:{dt_a} f={fill_a}",
                     lambda: S.clip(a_s, -1, 2), lambda: R.clip(a_r, -1, 2))
        return
    name = rng.choice(BINARY)
    if name == "power" and (np.dtype(dt_a).itemsize < 4 or np.dtype(dt_b).itemsize < 4 or "uint32" in (dt_a, dt_b)):
        name = "multiply"  # integer power in a narrow / unsigned type: outside the CUDA dtype matrix (TypeError)
    f = getattr(np, name)
    swap = rng.random() < 0.5
    desc = (f"#{i} np.{name}({fa}{base}:{dt_a} fill={fill_a}, {fb}{other}:{dt_b} fill={fill_b})"
            f"{' swapped' if swap else ''}")
    if swap:
        st.check("elemwise", desc, lambda: f(b_s, a_s), lambda: f(b_r, a_r))
    else:
        st.check("elemwise", desc, lambda: f(a_s, b_s), lambda: f(a_r, b_r))


REDUCE = ["sum", "prod", "max", "min", "any", "all", "mean", "var", "std", "nansum", "nanmax",
          "nanmin", "nanprod", "nanmean"]


def fam_reduce(rng, st, i):
    shape = draw_shape(rng, 1, 4)
    dt = rng.choice(DTYPES)
    fill = rng.choice([0, 0, 0, 1, 2]) if dt != "bool" else rng.choice([0, 0, 1])
    fmt = rng.choice(["coo", "coo", "gcxs"])
    name = rng.choice(REDUCE)
    if (np.dtype(dt).itemsize < 4 and name in ("sum", "nansum")) or name in ("prod", "nanprod"):
        fill = min(fill, 1)  # 2**n leaves int64 / is cast from float differently upstream (NumPy wraps)  # the reference multiplies / exponentiates the fill value IN the narrow dtype (wraps; NumPy does not)
    d = draw_dense(rng, shape, dt, fill=fill)
    if name.startswith("nan") and np.dtype(dt).kind == "f" and d.size and rng.random() < 0.7:
        d = d.copy()
        d[rng.random(shape) < 0.2] = np.nan
    x_s, x_r = both(d, fmt, fill=fill, rng=rng)
    nd = len(shape)
    r = rng.random()
    if r < 0.3:
        axis = None
    elif r < 0.7:
        axis = int(rng.integers(-nd, nd))
    else:
        k = int(rng.integers(1, nd + 1))
        axis = tuple(int(x) for x in rng.choice(nd, size=k, replace=False))
    kw = {"axis": axis}
    if name in ("argmax", "argmin"):
        if isinstance(axis, tuple):
            kw["axis"] = axis[0]
    if rng.random() < 0.4:
        kw["keepdims"] = True
    if name in ("sum", "prod", "mean", "var", "std", "nansum", "nanmean") and rng.random() < 0.3:
        kw["dtype"] = rng.choice(["float64", "float32"] + ([] if name in ("mean", "var", "std", "nanmean") else ["int64"]))
    if name in ("var", "std") and rng.random() < 0.4:
        kw["ddof"] = 1
    via = rng.choice(["func", "method", "numpy"])
    desc = f"#{i} {name}[{via}]({fmt}{shape}:{dt} fill={fill}, {kw})"
    exact = name not in ("mean", "var", "std", "nanmean")  # compositions: values to rounding, compared densely below

    def call(mod, x):
        if via == "method" and hasattr(x, name):
            return getattr(x, name)(**kw)
        if via == "numpy" and hasattr(np, name):
            return getattr(np, name)(x, **kw)
        return getattr(mod, name)(x, **kw)

    if exact:
        st.check("reduce", desc, lambda: call(S, x_s), lambda: call(R, x_r))
    else:
        st.n += 1
        got, want, es, er = run_pair(lambda: call(S, x_s), lambda: call(R, x_r))
        if es is not None or er is not None:
            if es is None and ref_crash(er):
                st.ref_crashes += 1
            elif (es is None) != (er is None):
                st.report("reduce", desc, f"error on one side only: here={es!r} reference={er!r}")
            elif type(es).__name__ != type(er).__name__ and not isinstance(es, type(er)):
                st.report("reduce", desc, f"error class: {type(es).__name__}({es}) != {type(er).__name__}({er})")
            return
        g = got.todense() if hasattr(got, "todense") else np.asarray(got)
        w = want.todense() if hasattr(want, "todense") else np.asarray(want)
        if type(got).__name__ != type(want).__name__ and (hasattr(got, "todense") or hasattr(want, "todense")):
            st.report("reduce", desc, f"class {type(got).__name__} != {type(want).__name__}")
        elif g.shape != w.shape or g.dtype != w.dtype:
            st.report("reduce", desc, f"shape/dtype {g.shape}:{g.dtype} != {w.shape}:{w.dtype}")
        elif not np.allclose(g, w, rtol=1e-5 if g.dtype == np.float32 else 1e-12, atol=1e-6 if g.dtype == np.float32 else 1e-12, equal_nan=True):
            try:  # the reference averages narrow integers IN their dtype (wraps); NumPy is the judge then
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    t = getattr(np, name)(d, **kw)
                if np.allclose(g, t, rtol=1e-5, atol=1e-6, equal_nan=True) and not np.allclose(w, t, rtol=1e-5, atol=1e-6, equal_nan=True):
                    st.ref_wrong += 1
                    return
            except Exception:  # noqa: BLE001
                pass
            st.report("reduce", desc, "values differ beyond rounding")


def fam_formats(rng, st, i):
    """Construction and format changes (SURVEY s8 rows a-1, a-2, a-19): COO from raw coords with duplicates / unsorted
    coords / explicit fill entries, GCXS with drawn compressed axes, transpose / reshape / change_compressed_axes /
    asformat round trips, broadcast_to."""
    shape = draw_shape(rng, 1, 4)
    dt = rng.choice(DTYPES)
    fill = rng.choice([0, 0, 1]) if dt != "bool" else rng.choice([0, 0, 1])
    nd = len(shape)
    what = rng.choice(["ctor", "gcxs_chain", "coo_chain", "broadcast_to", "getitem", "gcxs_raw"])
    if what == "gcxs_raw" and nd >= 2 and all(shape):
        # GCXS from raw (data, indices, indptr) with drawn compressed axes (the arrays come from the reference's own
        # conversion), then one consumer: tocoo / todense / transpose / a reduction / a product with a vector
        d = draw_dense(rng, shape, dt, fill=fill)
        k = int(rng.integers(1, nd))
        ca = tuple(sorted(int(x) for x in rng.choice(nd, size=k, replace=False)))
        g0 = R.COO.from_numpy(d, fill_value=np.asarray(fill, dtype=dt)[()]).asformat("gcxs", compressed_axes=ca)
        arrays = (g0.data.copy(), g0.indices.copy(), np.asarray(g0.indptr).copy())
        use = rng.choice(["tocoo", "todense", "T", "sum", "vec", "scipy"])

        def go(mod):
            g = mod.GCXS(arrays, shape=shape, compressed_axes=ca, fill_value=g0.fill_value)
            if use == "tocoo":
                return g.tocoo()
            if use == "todense":
                return g.todense()
            if use == "T":
                return g.T
            if use == "sum":
                return g.sum(axis=0)
            if use == "vec":
                if fill != 0:
                    return g.tocoo()
                return mod.tensordot(g, np.ones(shape[-1], dtype=np.float64), axes=1)
            if len(shape) == 2 and fill == 0 and np.dtype(dt).kind != "b":
                return mod.GCXS.from_scipy_sparse(g.to_scipy_sparse())
            return g

        st.check("formats", f"#{i} GCXS(raw arrays, shape={shape}, ca={ca}):{dt} fill={fill} -> {use}",
                 lambda: go(S), lambda: go(R))
        return
    if what == "gcxs_raw":
        what = "ctor"
    if what == "ctor":
        n = int(rng.integers(0, 12)) if all(shape) else 0
        coords = np.stack([rng.integers(0, max(s, 1), size=n) for s in shape]) if n else np.zeros((nd, 0), dtype=np.int64)
        data = (rng.integers(0 if np.dtype(dt).kind in "ub" else -3, 4, size=n)).astype(dt)
        kw = {}
        if rng.random() < 0.3:
            kw["prune"] = True
        if rng.random() < 0.3:
            kw["fill_value"] = np.asarray(fill, dtype=dt)[()]
        desc = f"#{i} COO(coords[{nd}x{n}], data:{dt}, shape={shape}, {kw})"
        st.check("formats", desc, lambda: S.COO(coords, data, shape=shape, **kw),
                 lambda: R.COO(coords, data, shape=shape, **kw))
        return
    d = draw_dense(rng, shape, dt, fill=fill)
    if what == "broadcast_to":
        lead = tuple(int(rng.integers(1, 4)) for _ in range(int(rng.integers(0, 3))))
        src = tuple(1 if rng.random() < 0.4 else s for s in shape)
        d2 = draw_dense(rng, src, dt, fill=fill)
        x_s, x_r = both(d2, "coo", fill=fill)
        target = lead + shape
        st.check("formats", f"#{i} broadcast_to(coo{src}:{dt} fill={fill}, {target})",
                 lambda: S.broadcast_to(x_s, target), lambda: R.broadcast_to(x_r, target))
        return
    # GCXS indexing is left out: upstream's result for None / negative-step indices is not NumPy's (axes land in
    # other positions), and indexing is not a row of SURVEY s8
    fmt = "gcxs" if what == "gcxs_chain" else ("coo" if what == "getitem" else rng.choice(["coo", "gcxs"]))
    x_s, x_r = both(d, fmt, fill=fill, rng=rng)
    if what == "getitem":
        idx = []
        for s in shape[: int(rng.integers(1, nd + 1))]:
            r = rng.random()
            if r < 0.35 and s:
                idx.append(int(rng.integers(-s, s)))
            elif r < 0.75:
                lo, hi = sorted(int(v) for v in rng.integers(-s - 1, s + 2, size=2))
                idx.append(slice(lo if rng.random() < 0.8 else None, hi if rng.random() < 0.8 else None,
                                 int(rng.choice([1, 1, 2, -1])) if rng.random() < 0.4 else None))
            elif r < 0.85:
                idx.append(None)
            elif r < 0.93 and Ellipsis not in idx:
                idx.append(Ellipsis)
            else:
                idx.append(slice(None))
        if rng.random() < 0.25 and shape[0]:
            # one integer-array index on the leading axis (the only advanced form upstream's COO takes: test_coo.py
            # test_advanced_indexing), possibly with repeats and negative entries
            idx[0] = [int(v) for v in rng.integers(-shape[0], shape[0], size=int(rng.integers(1, 5)))]
            idx = [v for v in idx if v is not None and v is not Ellipsis]
        idx = tuple(idx)
        st.check("formats", f"#{i} {fmt}{shape}:{dt} fill={fill} ca={getattr(x_r, 'compressed_axes', None)} [{idx}]",
                 lambda: x_s[idx], lambda: x_r[idx], truth=lambda: d[idx])  # negative steps: upstream != NumPy
        return
    steps = []
    for _ in range(int(rng.integers(1, 4))):
        op = rng.choice(["transpose", "reshape", "cca", "asformat", "T", "astype", "tocoo", "flatten"])
        if op == "transpose":
            steps.append(("transpose", tuple(int(v) for v in rng.permutation(nd))))
        elif op == "reshape":
            steps.append(("reshape", None))
        elif op == "cca":
            steps.append(("cca", None))
        elif op == "asformat":
            steps.append(("asformat", rng.choice(["coo", "gcxs"])))
        elif op == "astype":
            steps.append(("astype", rng.choice(["float64", "float32", "int64", "int32", "bool"])))
        else:
            steps.append((op, None))
    seed = int(rng.integers(1 << 30))

    def run(x, mod):
        r2 = np.random.default_rng(seed)
        for op, arg in steps:
            is_g = type(x).__name__ == "GCXS"
            if op == "transpose":
                if len(arg) == x.ndim:
                    x = x.transpose(arg)
            elif op == "reshape":
                n = int(np.prod(x.shape))
                cands = [(n,), (-1,)] + [(k, n // k) for k in (1, 2, 3, 4, 5, 6) if n and n % k == 0] + \
                        [(k, -1) for k in (2, 3) if n and n % k == 0] + [(1, n, 1)]
                x = x.reshape(cands[int(r2.integers(len(cands)))])
            elif op == "cca":
                if is_g and x.ndim >= 2:
                    k = int(r2.integers(1, x.ndim))
                    x = x.change_compressed_axes(tuple(sorted(int(v) for v in r2.choice(x.ndim, size=k, replace=False))))
            elif op == "asformat":
                x = x.asformat(arg)
            elif op == "T":
                x = x.T
            elif op == "astype":
                x = x.astype(arg)
            elif op == "tocoo":
                x = x.tocoo() if is_g else x
            elif op == "flatten":
                x = x.flatten()
        return x

    st.check("formats", f"#{i} {fmt}{shape}:{dt} fill={fill} ca={getattr(x_r, 'compressed_axes', None)} -> {steps} seed={seed}",
             lambda: run(x_s, S), lambda: run(x_r, R))


def fam_protocol(rng, st, i):
    """`__array_ufunc__` beyond the plain call (row a-17): ufunc.reduce, ufunc.outer, out=, in-place operators."""
    shape = draw_shape(rng, 1, 3, zero_ok=False)
    dt = rng.choice(FLOATS + ["int64", "int32"])
    fill = rng.choice([0, 0, 2])
    fmt = rng.choice(["coo", "gcxs"])
    d = draw_dense(rng, shape, dt, fill=fill)
    x_s, x_r = both(d, fmt, fill=fill, rng=rng)
    what = rng.choice(["reduce", "outer", "out", "inplace"])
    if what in ("out", "inplace") and fmt == "gcxs":
        # upstream's `out=` / in-place update of a GCXS array leaves a broken object behind (`_make_shallow_copy_of`
        # copies the COO result's attributes: no `_compressed_axes`), so there is nothing to compare with
        fmt = "coo"
        x_s, x_r = both(d, fmt, fill=fill)
    if what == "reduce":
        uf = getattr(np, rng.choice(["add", "multiply", "maximum", "minimum", "logical_and", "logical_or", "bitwise_or"]))
        if uf is np.multiply and fill > 1:
            uf = np.add  # fill ** n in the operand's narrow dtype wraps upstream
        if uf is np.bitwise_or and np.dtype(dt).kind == "f":
            uf = np.add
        axis = int(rng.integers(-len(shape), len(shape))) if rng.random() < 0.7 else None
        kw = {"axis": axis}
        if rng.random() < 0.3:
            kw["keepdims"] = True
        if rng.random() < 0.4:  # the method form, with the rest of the reduction op set
            uf2 = getattr(np, rng.choice(["fmax", "fmin", "maximum", "add", "logical_and", "logical_or"] +
                                         ([] if np.dtype(dt).kind == "f" else ["bitwise_and", "bitwise_xor"])))
            if uf2 is np.add and fill > 1:
                uf2 = np.maximum
            st.check("protocol", f"#{i} x.reduce(np.{uf2.__name__}, {kw}) x={fmt}{shape}:{dt} fill={fill}",
                     lambda: x_s.reduce(uf2, **kw), lambda: x_r.reduce(uf2, **kw))
            return
        st.check("protocol", f"#{i} np.{uf.__name__}.reduce({fmt}{shape}:{dt} fill={fill}, {kw})",
                 lambda: uf.reduce(x_s, **kw), lambda: uf.reduce(x_r, **kw))
    elif what == "outer":
        d2 = draw_dense(rng, draw_shape(rng, 1, 2, zero_ok=False), dt)
        y_s, y_r = both(d2, "coo")
        uf = getattr(np, rng.choice(["multiply", "add", "maximum"]))
        st.check("protocol", f"#{i} np.{uf.__name__}.outer({fmt}{shape}:{dt} fill={fill}, coo{d2.shape})",
                 lambda: uf.outer(x_s, y_s), lambda: uf.outer(x_r, y_r))
    elif what == "out":
        d2 = draw_dense(rng, shape, dt, fill=0)
        y_s, y_r = both(d2, fmt, rng=None)
        odt = rng.choice([dt, "float64", "float32"])
        o_s, o_r = both(np.zeros(shape, dtype=odt), fmt)
        uf = getattr(np, rng.choice(["add", "multiply", "subtract"]))

        def go(a, b, o):
            r = uf(a, b, out=o)
            assert r is o
            return r

        st.check("protocol", f"#{i} np.{uf.__name__}({fmt}{shape}:{dt} fill={fill}, {fmt}, out={fmt}:{odt})",
                 lambda: go(x_s, y_s, o_s), lambda: go(x_r, y_r, o_r))
    else:
        d2 = draw_dense(rng, tuple(s if rng.random() < 0.7 else 1 for s in shape), dt)
        y_s, y_r = both(d2, rng.choice(["coo", "dense"]))
        opn = rng.choice(["iadd", "imul", "isub"])
        import operator

        def go(a, b):
            a = a.copy() if hasattr(a, "copy") else a
            return getattr(operator, opn)(a, b)

        st.check("protocol", f"#{i} {opn}({fmt}{shape}:{dt} fill={fill}, {type(y_r).__name__}{d2.shape})",
                 lambda: go(x_s, y_s), lambda: go(x_r, y_r))


def fam_scipy(rng, st, i):
    """scipy.sparse operands (2-D) next to COO / GCXS / ndarray in the products and in element-wise calls
    (_common.py:127-130, _umath.py:432-433), non-zero fill values in products (error parity), COO built with the
    `sorted=False` / `has_duplicates=True` flags and 32-bit coordinates feeding a product."""
    import scipy.sparse as ss

    M, K, N = (int(v) for v in rng.integers(1, 6, size=3))
    dt_a, dt_b = rng.choice(FLOATS + ["int64", "int32"]), rng.choice(FLOATS + ["int64"])
    da, db = draw_dense(rng, (M, K), dt_a), draw_dense(rng, (K, N), dt_b)
    mk = {"csr": ss.csr_array, "csc": ss.csc_array, "coo": ss.coo_array, "csr_matrix": ss.csr_matrix}
    what = rng.choice(["dot_scipy", "ew_scipy", "fill_error", "flags"])
    if what == "dot_scipy":
        ka = rng.choice(list(mk))
        fb = rng.choice(["coo", "gcxs", "dense", "scipy"])
        a = mk[ka](da)
        if fb == "scipy":
            b_s = b_r = mk[rng.choice(list(mk))](db)
        else:
            b_s, b_r = both(db, fb, rng=rng)
        swap = rng.random() < 0.4 and fb != "scipy"
        fn = rng.choice(["tensordot", "matmul", "dot"])
        if swap:  # (K,N)^T x ... keep shapes compatible: b^T (N,K) @ a^T (K,M)
            a = mk[ka](np.ascontiguousarray(da.T))
            b2_s, b2_r = both(np.ascontiguousarray(db.T), fb, rng=rng)
            args_s, args_r = (b2_s, a), (b2_r, a)
        else:
            args_s, args_r = (a, b_s), (a, b_r)
        kw = {"axes": 1} if fn == "tensordot" else {}
        st.check("scipy", f"#{i} {fn}({'x,' if swap else ''}scipy.{ka}({M},{K}):{dt_a}{'' if swap else ',x'}) x={fb}:{dt_b}",
                 lambda: getattr(S, fn)(*args_s, **kw), lambda: getattr(R, fn)(*args_r, **kw))
    elif what == "ew_scipy":
        d2 = draw_dense(rng, (M, K), dt_b)
        sc = mk[rng.choice(list(mk))](d2)
        fa = rng.choice(["coo", "gcxs"])
        x_s, x_r = both(da, fa, rng=rng)
        name = rng.choice(["add", "multiply", "maximum", "subtract", "greater"])
        f = getattr(np, name)
        st.check("scipy", f"#{i} elemwise(np.{name}, {fa}({M},{K}):{dt_a}, scipy:{dt_b})",
                 lambda: S.elemwise(f, x_s, sc), lambda: R.elemwise(f, x_r, sc))
    elif what == "fill_error":
        fa, fb = rng.choice(["coo", "gcxs"]), rng.choice(["coo", "gcxs", "dense"])
        fill_a, fill_b = rng.choice([0, 1, 2]), rng.choice([0, 0, 3])
        a_s, a_r = both(draw_dense(rng, (M, K), dt_a, fill=fill_a), fa, fill=fill_a, rng=rng)
        b_s, b_r = both(draw_dense(rng, (K, N), dt_b, fill=fill_b), fb, fill=fill_b, rng=rng)
        fn = rng.choice(["tensordot", "matmul", "dot"])
        kw = {"axes": 1} if fn == "tensordot" else {}
        st.check("scipy", f"#{i} {fn}({fa} fill={fill_a}, {fb} fill={fill_b})",
                 lambda: getattr(S, fn)(a_s, b_s, **kw), lambda: getattr(R, fn)(a_r, b_r, **kw))
    else:
        n = int(rng.integers(0, 14))
        idt = rng.choice(["int64", "int32", "uint8"])
        coords = np.stack([rng.integers(0, M, size=n), rng.integers(0, K, size=n)]).astype(idt)
        data = rng.integers(-3, 4, size=n).astype(dt_a)
        mode = rng.choice(["plain", "dups", "unsorted_ok"])
        if mode == "unsorted_ok":  # unique coordinates in random order, flags say so
            flat = rng.choice(M * K, size=min(n, M * K), replace=False)
            coords = np.stack(np.unravel_index(flat, (M, K))).astype(idt)
            data = data[: coords.shape[1]]
            kw = {"has_duplicates": False, "sorted": False}
        elif mode == "dups":
            kw = {"has_duplicates": True, "sorted": False}
        else:
            kw = {}
        fb = rng.choice(["coo", "gcxs", "dense"])
        b_s, b_r = both(db, fb, rng=rng)
        st.check("scipy", f"#{i} COO(coords:{idt}[2x{coords.shape[1]}], {kw}) ({M},{K}):{dt_a} @ {fb}:{dt_b}",
                 lambda: S.COO(coords, data, shape=(M, K), **kw) @ b_s,
                 lambda: R.COO(coords, data, shape=(M, K), **kw) @ b_r, truth=None)


def fam_einsum(rng, st, i):
    """`einsum` (the MTTKRP example's call, examples/mttkrp_example.py upstream): random subscripts over 1-3 operands,
    repeated indices inside an operand included, explicit and implicit outputs, COO / GCXS / dense operands."""
    letters = "ijkl"
    sizes = {c: int(rng.integers(1, max(5, MAX_EXTENT[0] - 1))) for c in letters}
    n_ops = int(rng.integers(1, 4))
    subs, ops_s, ops_r, descs = [], [], [], []
    dt = rng.choice(FLOATS + ["int64"])
    for k in range(n_ops):
        nd = int(rng.integers(1, 4))
        sub = "".join(rng.choice(list(letters), size=nd, replace=rng.random() < 0.15))
        shape = tuple(sizes[c] for c in sub)
        fmt = rng.choice(["coo", "coo", "gcxs", "dense"]) if (k or n_ops > 1) else rng.choice(["coo", "gcxs"])
        d = draw_dense(rng, shape, dt)
        a_s, a_r = both(d, fmt, rng=rng)
        subs.append(sub), ops_s.append(a_s), ops_r.append(a_r), descs.append(f"{fmt}{shape}")
    if not any(isinstance(o, R.SparseArray) for o in ops_r):
        ops_s[0], ops_r[0] = both(np.asarray(ops_r[0]), "coo")
    used = sorted(set("".join(subs)))
    expr = ",".join(subs)
    if rng.random() < 0.7:
        k = int(rng.integers(0, len(used) + 1))
        out = "".join(rng.permutation(used)[:k])
        expr += "->" + out
    kw = {}
    if rng.random() < 0.15:
        kw["dtype"] = rng.choice(["float64", "float32"])
    if rng.random() < 0.25 and isinstance(ops_r[0], R.SparseArray) and not kw:
        st.check("einsum", f"#{i} np.einsum('{expr}', {', '.join(descs)}) :{dt}",
                 lambda: np.einsum(expr, *ops_s), lambda: np.einsum(expr, *ops_r))
        return
    st.check("einsum", f"#{i} einsum('{expr}', {', '.join(descs)}) :{dt} {kw}",
             lambda: S.einsum(expr, *ops_s, **kw), lambda: R.einsum(expr, *ops_r, **kw))


def fam_helpers(rng, st, i):
    """Row a-22: `equivalent` (bit-pattern equality with NaN == NaN, +0.0 != -0.0), `check_zero_fill_value`,
    `normalize_axis`, `_dot_dtype` -- called directly on both sides."""
    from sparse.numba_backend import _utils as RU
    from sparse_b200 import _utils as SU

    pool = [0.0, -0.0, 1.0, np.nan, -np.nan, np.inf, -np.inf, 2, 0, True, False, np.float32("nan"), np.float32(-0.0),
            np.int8(0), np.uint8(3), np.float32(1.5), 1.5]
    what = rng.choice(["equivalent", "czfv", "normalize_axis"])
    if what == "equivalent":
        def pick():
            if rng.random() < 0.5:
                return pool[int(rng.integers(len(pool)))]
            dt = rng.choice(["float64", "float32", "int64", "bool"])
            vals = [pool[int(rng.integers(len(pool)))] for _ in range(int(rng.integers(1, 5)))]
            with np.errstate(all="ignore"):
                return np.array([0 if (isinstance(v, float) and v != v and dt in ("int64", "bool")) or
                                 (isinstance(v, (float, np.floating)) and np.isinf(v) and dt in ("int64", "bool")) else v
                                 for v in vals]).astype(dt)
        x, y = pick(), pick()
        if np.ndim(x) and np.ndim(y) and np.shape(x) != np.shape(y):
            y = np.resize(y, np.shape(x))
        loose = bool(rng.random() < 0.5)
        st.check("helpers", f"#{i} equivalent({x!r}, {y!r}, loose={loose})",
                 lambda: np.asarray(SU.equivalent(x, y, loose=loose)), lambda: np.asarray(RU.equivalent(x, y, loose=loose)))
    elif what == "czfv":
        fills = [pool[int(rng.integers(len(pool)))] for _ in range(int(rng.integers(1, 3)))]
        dts = [rng.choice(["float64", "float32", "int64"]) for _ in fills]
        def mk(mod):
            out = []
            for f, dt in zip(fills, dts):
                with np.errstate(all="ignore"):
                    fv = np.asarray(f).astype(dt)[()] if not (np.asarray(f).dtype.kind == "f" and not np.isfinite(f) and dt == "int64") else np.int64(1)
                out.append(mod.COO.from_numpy(np.full((2, 2), fv, dtype=dt), fill_value=fv))
            return out
        loose = bool(rng.random() < 0.7)
        st.check("helpers", f"#{i} check_zero_fill_value(fills={fills} as {dts}, loose={loose})",
                 lambda: SU.check_zero_fill_value(*mk(S), loose=loose), lambda: RU.check_zero_fill_value(*mk(R), loose=loose))
    else:
        nd = int(rng.integers(1, 5))
        r = rng.random()
        if r < 0.3:
            axis = int(rng.integers(-nd - 1, nd + 1))
        elif r < 0.7:
            axis = tuple(int(v) for v in rng.integers(-nd - 1, nd + 1, size=int(rng.integers(0, 4))))
        elif r < 0.8:
            axis = None
        elif r < 0.9:
            axis = [int(v) for v in rng.integers(-nd, nd, size=2)]
        else:
            axis = rng.choice([1.5, "x"])
            axis = float(axis) if axis == "1.5" else str(axis)
        st.check("helpers", f"#{i} normalize_axis({axis!r}, {nd})",
                 lambda: np.asarray(SU.normalize_axis(axis, nd), dtype=object), lambda: np.asarray(RU.normalize_axis(axis, nd), dtype=object))


def fam_io(rng, st, i):
    """Row f-4: .npz files cross the two packages in both directions (compressed or not, COO and GCXS, fill values)."""
    import tempfile

    shape = draw_shape(rng, 1, 4)
    dt = rng.choice(DTYPES)
    fill = rng.choice([0, 0, 1]) if dt != "bool" else rng.choice([0, 1])
    # a 1-D GCXS array is stored with `compressed_axes=None`, an object array: upstream cannot load such a file back
    # (allow_pickle=False), nor can this package -- same file, same refusal, nothing to compare
    fmt = rng.choice(["coo", "gcxs"]) if len(shape) > 1 else "coo"
    d = draw_dense(rng, shape, dt, fill=fill)
    x_s, x_r = both(d, fmt, fill=fill, rng=rng)
    comp = bool(rng.random() < 0.5)
    with tempfile.TemporaryDirectory() as tmp:
        f1, f2 = os.path.join(tmp, "a.npz"), os.path.join(tmp, "b.npz")
        R.save_npz(f1, x_r, compressed=comp)
        st.check("io", f"#{i} load_npz(here) of the reference's file: {fmt}{shape}:{dt} fill={fill} compressed={comp}",
                 lambda: S.load_npz(f1), lambda: x_r)
        S.save_npz(f2, x_s, compressed=comp)
        st.check("io", f"#{i} the reference loads this package's file: {fmt}{shape}:{dt} fill={fill}",
                 lambda: x_s, lambda: R.load_npz(f2))


def fam_fused(rng, st, i):
    """Rows a-20 / a-21: the fused SDDMM / MTTKRP entry points AND the unfused example expressions
    (`s * (a @ b)`, examples/sddmm_example.py:52; `sum(B[..., None] * D[None, None] * C[None, :, None], axis=(1, 2))`,
    examples/mttkrp_example.py:52) against the reference evaluating the example expression.  Integer-valued floats:
    every order of summation gives the same bits, so the comparison is exact."""
    dt = rng.choice(FLOATS)
    if rng.random() < 0.5:
        M, K, N = (int(v) for v in rng.integers(1, 7, size=3))
        fmt = rng.choice(["coo", "gcxs"])
        ds = draw_dense(rng, (M, N), dt)
        a, b = draw_dense(rng, (M, K), dt, density=1.0), draw_dense(rng, (K, N), dt, density=1.0)
        s_s, s_r = both(ds, fmt, rng=rng)
        fused = rng.random() < 0.5
        st.check("fused", f"#{i} {'sddmm(s,a,b)' if fused else 's * (a @ b)'} s={fmt}({M},{N}) K={K} :{dt}",
                 (lambda: S.sddmm(s_s, a, b)) if fused else (lambda: s_s * (a @ b)), lambda: s_r * (a @ b))
    else:
        I, Kk, L, J = (int(v) for v in rng.integers(1, 6, size=4))
        fmt = rng.choice(["coo", "gcxs"])
        dB = draw_dense(rng, (I, Kk, L), dt)
        Dm, Cm = draw_dense(rng, (L, J), dt, density=1.0), draw_dense(rng, (Kk, J), dt, density=1.0)
        B_s, B_r = both(dB, fmt, rng=rng)
        fused = rng.random() < 0.5

        def expr(mod, B):
            return mod.sum(B[:, :, :, None] * Dm[None, None, :, :] * Cm[None, :, None, :], axis=(1, 2))

        if fmt == "gcxs":  # upstream's GCXS indexing with None is not NumPy's (DESIGN s4): give both sides COO there
            B_r = B_r.tocoo()
            B_s2 = B_s.tocoo()
        else:
            B_s2 = B_s
        want = lambda: expr(R, B_r)  # noqa: E731
        if fused:
            # the fused kernel returns the format of B; the expression's result is compared densely
            st.n += 1
            got, w, es, er = run_pair(lambda: S.mttkrp(B_s, Dm, Cm), want)
            if es is not None or er is not None:
                st.report("fused", f"#{i} mttkrp", f"raised: here={es!r} reference={er!r}")
            elif not arr_eq(got.todense(), w.todense()) or got.dtype != w.dtype:
                st.report("fused", f"#{i} mttkrp(B={fmt}({I},{Kk},{L}), J={J}) :{dt}", "values / dtype differ")
        else:
            st.check("fused", f"#{i} mttkrp expression B={fmt}({I},{Kk},{L}) J={J} :{dt}", lambda: expr(S, B_s2), want)


def fam_special(rng, st, i):
    """NaN / +-inf / -0.0 in the data AND as fill values (float operands): element-wise binary / unary calls and
    reductions.  Pruning is by bit pattern upstream, NaN fills equal themselves, -0.0 is not +0.0."""
    specials = [np.nan, np.inf, -np.inf, -0.0, 0.0]
    dt_a, dt_b = rng.choice(FLOATS), rng.choice(FLOATS + ["int64"])
    shape = draw_shape(rng, 1, 3, zero_ok=False)

    def arr(shape, dt, fill):
        d = draw_dense(rng, shape, dt, fill=0).astype(dt)
        if np.dtype(dt).kind == "f":
            d[d == 0] = fill
            for v in specials:
                d[rng.random(shape) < 0.08] = v
        return d

    fill_a = float(rng.choice(specials + [0.0, 0.0, 2.0]))
    da = arr(shape, dt_a, fill_a)
    fmt = rng.choice(["coo", "gcxs"])
    fv = np.asarray(fill_a, dtype=dt_a)[()]
    a_r, a_s = R.COO.from_numpy(da, fill_value=fv), S.COO.from_numpy(da, fill_value=fv)
    if fmt == "gcxs":
        a_r, a_s = a_r.asformat("gcxs"), a_s.asformat("gcxs")
    mode = rng.choice(["binary", "binary", "scalar", "unary", "reduce"])
    if mode == "unary":
        name = rng.choice(["negative", "abs", "sign", "isnan", "isinf", "isfinite", "signbit", "square", "sqrt", "floor",
                           "exp", "log1p", "reciprocal"])
        f = getattr(np, name)
        st.check("special", f"#{i} np.{name}({fmt}{shape}:{dt_a} fill={fill_a})", lambda: f(a_s), lambda: f(a_r))
    elif mode == "scalar":
        name = rng.choice(["add", "multiply", "maximum", "minimum", "fmax", "fmin", "greater", "equal", "not_equal",
                           "true_divide", "subtract"])
        f = getattr(np, name)
        sc = rng.choice(specials + [1.0, 2.0])
        if sc == 0 and name in ("maximum", "minimum", "fmax", "fmin"):
            sc = 1.0  # (+0.0, -0.0) ties: NumPy's answer depends on the loop, see the binary branch
        left = rng.random() < 0.5
        st.check("special", f"#{i} np.{name}({'sc,' if left else ''}{fmt}{shape}:{dt_a} fill={fill_a}{'' if left else ',sc'}) sc={sc}",
                 (lambda: f(sc, a_s)) if left else (lambda: f(a_s, sc)), (lambda: f(sc, a_r)) if left else (lambda: f(a_r, sc)))
    elif mode == "binary":
        other = tuple(s_ if rng.random() < 0.7 else 1 for s_ in shape)
        fill_b = float(rng.choice(specials + [0.0, 0.0, 3.0])) if np.dtype(dt_b).kind == "f" else int(rng.choice([0, 0, 1]))
        db = arr(other, dt_b, fill_b) if np.dtype(dt_b).kind == "f" else draw_dense(rng, other, dt_b, fill=fill_b)
        fb = rng.choice(["coo", "gcxs", "dense"])
        b_s, b_r = both(db, fb, fill=fill_b, rng=rng)
        # maximum / minimum / fmax / fmin stay out of THIS family's binary draws: on a (+0.0, -0.0) pair NumPy's own
        # answer depends on the loop (SIMD body, scalar tail and scalar call disagree), so there is no bit pattern to
        # reproduce; they are exercised with special scalars above and with ordinary values in fam_elemwise
        name = rng.choice(["add", "subtract", "multiply", "true_divide", "greater",
                           "less_equal", "equal", "not_equal", "logical_and", "logical_or", "logical_xor"])
        f = getattr(np, name)
        st.check("special", f"#{i} np.{name}({fmt}{shape}:{dt_a} fill={fill_a}, {fb}{other}:{dt_b} fill={fill_b})",
                 lambda: f(a_s, b_s), lambda: f(a_r, b_r))
    else:
        name = rng.choice(["sum", "prod", "max", "min", "nansum", "nanmax", "nanmin", "nanprod", "any", "all"])
        axis = int(rng.integers(-len(shape), len(shape))) if rng.random() < 0.7 else None
        kw = {"axis": axis, **({"keepdims": True} if rng.random() < 0.3 else {})}

        def call(mod, x):
            return getattr(mod, name)(x, **kw)

        # sums / products of special values: order-independent only as sets of bits up to NaN payload -- compared
        # exactly anyway (inf + -inf = NaN on both sides; NumPy pairwise vs sequential never differs on these inputs)
        # a sum / product that turns into NaN carries a sign / payload that depends on the order of the operations
        # (inf + -inf is the negative default NaN on x86, NaN + x keeps the first payload); upstream compares bit
        # patterns, so WHICH NaN results equal a NaN fill value -- and are pruned -- is order-dependent: dense compare
        st.check("special", f"#{i} {name}({fmt}{shape}:{dt_a} fill={fill_a}, {kw})", lambda: call(S, a_s), lambda: call(R, a_r),
                 exact_layout=name not in ("sum", "prod", "nansum", "nanprod"))


def fam_where(rng, st, i):
    """Three-argument `where` with every operand drawn independently: COO / GCXS / ndarray in each slot, 0-D and
    zero-length operands, broadcasting between all three, non-zero fill values.  Upstream's one elemwise call decides
    sparse-vs-dense (and the error) on where(fills | ndarrays); the result format follows the sparse operands."""
    base = draw_shape(rng, 0, 3)

    def operand(kinds, dts, fills):
        shape = tuple(s if rng.random() < 0.7 else 1 for s in base)
        shape = shape[int(rng.integers(0, len(shape) + 1)):]
        dt, fill, fmt = rng.choice(dts), rng.choice(fills), rng.choice(kinds)
        d = draw_dense(rng, shape, dt, fill=fill)
        return both(d, fmt, fill=fill, rng=rng) + (f"{fmt}{shape}:{dt} f={fill}",)

    c_s, c_r, dc = operand(["coo", "coo", "gcxs", "dense"], ["bool", "float32", "int64"], [0, 0, 1])
    x_s, x_r, dx = operand(["coo", "gcxs", "dense"], ["float64", "float32", "int64"], [0, 0, 2])
    y_s, y_r, dy = operand(["coo", "gcxs", "dense"], ["float64", "float32", "int64"], [0, 0, 3])
    if not any(isinstance(v, R.SparseArray) for v in (c_r, x_r, y_r)):
        c_s, c_r = both(np.asarray(c_r), "coo")
    via = "numpy" if rng.random() < 0.3 and isinstance(c_r, R.SparseArray) else "func"  # np.where: __array_function__
    st.check("where", f"#{i} where({dc}, {dx}, {dy}) via={via}", (lambda: S.where(c_s, x_s, y_s)) if via == "func" else (lambda: np.where(c_s, x_s, y_s)),
             (lambda: R.where(c_r, x_r, y_r)) if via == "func" else (lambda: np.where(c_r, x_r, y_r)))


NARY = {"x*y+z": lambda x, y, z: x * y + z, "(x+y)*z": lambda x, y, z: (x + y) * z,
        "max(x,y)-z": lambda x, y, z: np.maximum(x, y) - z, "x*y": lambda x, y: x * y, "x+y": lambda x, y: x + y,
        "x*(y>z)": lambda x, y, z: x * (y > z)}


def fam_nary(rng, st, i):
    """User-defined functions through `elemwise` with every operand drawn independently (COO / GCXS / ndarray, 0-D and
    zero-length operands, non-zero fill values, broadcasting between all of them): upstream evaluates the function on
    matched data and decides sparse-or-dense on one probe; the operator-by-operator evaluation here has to agree in
    class, fill value and the exact stored set (signed zeros included)."""
    base = draw_shape(rng, 0, 3)
    name = rng.choice(list(NARY))
    f = NARY[name]
    ops_s, ops_r, descs = [], [], []
    for _ in range(f.__code__.co_argcount):
        shape = tuple(s if rng.random() < 0.7 else 1 for s in base)
        shape = shape[int(rng.integers(0, len(shape) + 1)):]
        dt, fill, fmt = rng.choice(["float64", "float32", "int64"]), rng.choice([0, 0, 2]), rng.choice(["coo", "gcxs", "dense"])
        a, b = both(draw_dense(rng, shape, dt, fill=fill), fmt, fill=fill, rng=rng)
        ops_s.append(a), ops_r.append(b), descs.append(f"{fmt}{shape}:{dt} f={fill}")
    if not any(isinstance(v, R.SparseArray) for v in ops_r):
        ops_s[0], ops_r[0] = both(np.asarray(ops_r[0]), "coo")
    st.check("nary", f"#{i} elemwise({name}; {', '.join(descs)})", lambda: S.elemwise(f, *ops_s),
             lambda: R.elemwise(f, *ops_r))


def fam_methods(rng, st, i):
    """Methods and properties next to the path: astype (casting / copy, values that collapse onto the fill value,
    0-D arrays), real / imag / conj / T, COO and GCXS constructors in their argument forms, linear_loc / nonzero /
    flatten / squeeze / swapaxes."""
    shape = draw_shape(rng, 0, 3)
    dt = rng.choice(DTYPES)
    fill = int(rng.choice([0, 0, 1, 2])) if dt != "bool" else int(rng.choice([0, 1]))
    d = draw_dense(rng, shape, dt, fill=fill)
    what = rng.choice(["astype", "attr", "coo_ctor", "gcxs_ctor", "helper"])
    if what == "astype":
        if np.dtype(dt).kind == "f" and d.size and rng.random() < 0.3:
            d = d.copy()
            d[rng.random(shape) < 0.3] = rng.choice([0.4, -0.6, 1e-50, 3e9, np.nan])
        fmt = rng.choice(["coo", "gcxs"])
        x_s, x_r = both(d, fmt, fill=fill, rng=rng)
        to, kw = rng.choice(DTYPES), {}
        if rng.random() < 0.3:
            kw["casting"] = rng.choice(["safe", "same_kind", "unsafe", "no", "equiv"])
        if rng.random() < 0.3:
            kw["copy"] = bool(rng.random() < 0.5)
        st.check("methods", f"#{i} {fmt}{shape}:{dt} f={fill} .astype({to}, {kw})",
                 lambda: x_s.astype(to, **kw), lambda: x_r.astype(to, **kw))
    elif what == "attr":
        fmt = rng.choice(["coo", "gcxs"])
        x_s, x_r = both(d, fmt, fill=fill, rng=rng)
        attr = rng.choice(["real", "imag", "conj()", "T", "mT" if len(shape) >= 2 else "T", "nbytes", "density", "nnz"])
        if attr == "nbytes" and (fmt == "gcxs" and len(shape) < 2):
            attr = "nnz"  # upstream's nbytes of a 0-D / 1-D GCXS array raises (indptr is a tuple there)

        def get(x):
            v = x.conj() if attr == "conj()" else getattr(x, attr)
            return np.asarray(v) if attr in ("nbytes", "density", "nnz") else v

        st.check("methods", f"#{i} {fmt}{shape}:{dt} f={fill} .{attr}", lambda: get(x_s), lambda: get(x_r))
    elif what == "coo_ctor":
        nd = max(1, len(shape))
        shp = tuple(max(1, s) for s in (shape or (3,)))[:nd]
        n = int(rng.integers(0, 8))
        coords = np.stack([rng.integers(0, s, size=n) for s in shp])
        data = rng.integers(0 if dt == "bool" else -3, 4, size=n).astype(dt)
        mode = rng.choice(["list", "noshape", "scalar_data", "1d", "copy_of", "fill", "prune_false", "dups", "idx_dtype"])
        kw = {"shape": shp}
        args = (coords, data)
        if mode == "list":
            args = (coords.tolist(), data.tolist())
        elif mode == "noshape":
            kw = {}
        elif mode == "scalar_data":
            args = (coords, np.dtype(dt).type(2))
        elif mode == "1d":
            kw, args = {"shape": (shp[0],)}, (coords[0], data)
        elif mode == "fill":
            kw["fill_value"] = np.dtype(dt).type(1)
        elif mode == "prune_false":
            kw["prune"] = False
        elif mode == "dups":
            kw["has_duplicates"] = True
        elif mode == "idx_dtype":
            kw["idx_dtype"] = rng.choice([np.int32, np.uint8, np.int64])
        if mode == "copy_of":
            st.check("methods", f"#{i} COO(COO) {shp}:{dt}", lambda: S.COO(S.COO(coords, data, shape=shp)),
                     lambda: R.COO(R.COO(coords, data, shape=shp)))
        else:
            st.check("methods", f"#{i} COO[{mode}] n={n} {shp}:{dt}", lambda: S.COO(*args, **kw), lambda: R.COO(*args, **kw))
    elif what == "gcxs_ctor":
        if not shape:
            shape, d = (3,), draw_dense(rng, (3,), dt, fill=fill)
        nd, kw = len(shape), {}
        if nd >= 2 and rng.random() < 0.6:
            k = int(rng.integers(1, nd))
            kw["compressed_axes"] = tuple(sorted(int(x) for x in rng.choice(nd, size=k, replace=False)))
        fv = np.asarray(fill, dtype=dt)[()]
        mode = rng.choice(["from_numpy", "from_coo", "ctor_coo", "ctor_nd", "ctor_gcxs"])
        if mode == "from_numpy":
            st.check("methods", f"#{i} GCXS.from_numpy({shape}:{dt}, {kw})", lambda: S.GCXS.from_numpy(d, **kw),
                     lambda: R.GCXS.from_numpy(d, **kw))
        elif mode == "from_coo":
            st.check("methods", f"#{i} GCXS.from_coo({shape}:{dt} f={fill}, {kw})",
                     lambda: S.GCXS.from_coo(S.COO.from_numpy(d, fill_value=fv), **kw),
                     lambda: R.GCXS.from_coo(R.COO.from_numpy(d, fill_value=fv), **kw))
        elif mode == "ctor_coo":
            st.check("methods", f"#{i} GCXS(coo {shape}:{dt} f={fill}, {kw})",
                     lambda: S.GCXS(S.COO.from_numpy(d, fill_value=fv), **kw),
                     lambda: R.GCXS(R.COO.from_numpy(d, fill_value=fv), **kw))
        elif mode == "ctor_nd":
            st.check("methods", f"#{i} GCXS(ndarray {shape}:{dt}, {kw})", lambda: S.GCXS(d, **kw), lambda: R.GCXS(d, **kw))
        else:
            st.check("methods", f"#{i} GCXS(GCXS {shape}:{dt}, {kw})", lambda: S.GCXS(S.GCXS.from_numpy(d), **kw),
                     lambda: R.GCXS(R.GCXS.from_numpy(d), **kw))
    else:
        if not shape:
            shape, d = (4,), draw_dense(rng, (4,), dt, fill=0)
        x_s, x_r = both(draw_dense(rng, shape, dt), "coo")
        m = rng.choice(["linear_loc", "nonzero", "flatten", "squeeze", "swapaxes"])

        def call(x):
            if m == "linear_loc":
                return np.asarray(x.linear_loc())
            if m == "nonzero":
                return np.stack([np.asarray(v) for v in x.nonzero()])
            return x.flatten() if m == "flatten" else x.squeeze() if m == "squeeze" else x.swapaxes(0, -1)

        st.check("methods", f"#{i} coo{shape}:{dt} .{m}()", lambda: call(x_s), lambda: call(x_r))


def fam_join(rng, st, i):
    """kron (row 7 / the round-1 advisor item: stored x stored only), concatenate and stack (the N-D matmul is built on
    stack): formats, fill values, zero-length pieces, narrow integer dtypes."""
    what = rng.choice(["kron", "concatenate", "stack"])
    dt = rng.choice(["float64", "float32", "int64", "int8", "bool"])
    if what == "kron":
        sa, sb = draw_shape(rng, 1, 3, zero_ok=False), draw_shape(rng, 1, 3, zero_ok=False)
        da, db = draw_dense(rng, sa, dt), draw_dense(rng, sb, rng.choice(["float64", "int64", dt]))
        fa, fb = rng.choice(["coo", "gcxs", "dense"]), rng.choice(["coo", "gcxs", "dense"])
        if fa == "dense" and fb == "dense":
            fa = "coo"
        a_s, a_r = both(da, fa, rng=rng)
        b_s, b_r = both(db, fb, rng=rng)
        st.check("join", f"#{i} kron({fa}{sa}:{da.dtype}, {fb}{sb}:{db.dtype})", lambda: S.kron(a_s, b_s),
                 lambda: R.kron(a_r, b_r))
        return
    base = draw_shape(rng, 1, 3)
    k, axis = int(rng.integers(1, 4)), int(rng.integers(-len(base), len(base)))
    fill = int(rng.choice([0, 0, 2])) if dt != "bool" else 0
    fmt = rng.choice(["coo", "gcxs"])
    arrs_s, arrs_r = [], []
    for _ in range(k):
        shp = list(base)
        if what == "concatenate":
            shp[axis] = int(rng.integers(0, 4))
        a, b = both(draw_dense(rng, tuple(shp), dt, fill=fill), fmt, fill=fill, rng=rng)
        arrs_s.append(a), arrs_r.append(b)
    st.check("join", f"#{i} {what}({k} x {fmt}{base}:{dt} f={fill}, axis={axis})",
             lambda: getattr(S, what)(arrs_s, axis=axis), lambda: getattr(R, what)(arrs_r, axis=axis))


FAMILIES = {"join": fam_join, "methods": fam_methods, "nary": fam_nary, "where": fam_where, "special": fam_special, "fused": fam_fused, "io": fam_io, "helpers": fam_helpers, "einsum": fam_einsum, "scipy": fam_scipy, "dot": fam_dot, "elemwise": fam_elemwise, "reduce": fam_reduce, "formats": fam_formats,
            "protocol": fam_protocol}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", type=int, default=3000)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--family", default="all")
    ap.add_argument("--only", type=int, default=-1, help="re-run one case index")
    ap.add_argument("--max-extent", type=int, default=6, help="axis lengths are drawn below this (default 6)")
    ap.add_argument("-v", action="store_true")
    args = ap.parse_args()
    MAX_EXTENT[0] = args.max_extent
    fams = list(FAMILIES) if args.family == "all" else args.family.split(",")
    st = Stats(args.v)
    for fam in fams:
        for i in range(args.cases):
            if args.only >= 0 and i != args.only:
                continue
            rng = np.random.default_rng([args.seed, i, sum(map(ord, fam))])
            try:
                FAMILIES[fam](rng, st, i)
            except Exception as e:  # noqa: BLE001  (a bug of the fuzzer itself or of input construction)
                st.report(fam, f"#{i}", f"fuzzer/construct error {type(e).__name__}: {e}\n" +
                          "".join(traceback.format_exception(type(e), e, e.__traceback__)[-4:]))
        print(f"== {fam}: {st.n} comparisons so far, {st.bad} mismatches, {st.errs_both} raised on both sides", flush=True)
    print("\nmismatch classes:")
    for (fam, k), v in sorted(st.kinds.items(), key=lambda kv: -kv[1]):
        print(f"  {v:5d}  [{fam}] {k}")
    print(f"TOTAL {st.n} comparisons, {st.bad} mismatches ({st.errs_both} raised the same error class on both sides, "
          f"{st.ref_crashes} crashed inside the reference only, {st.ref_wrong} reference results contradicted by NumPy)")
    return 1 if st.bad else 0


if __name__ == "__main__":
    sys.exit(main())
