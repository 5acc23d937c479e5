"""sparse_b200 -- a B200-native (sm_100a) implementation of pydata/sparse's data-parallel hot path.

Drop-in names for that path: ``COO``, ``GCXS`` (``CSR``/``CSC``), ``tensordot``, ``matmul``, ``dot``,
``elemwise``, reductions (``sum``/``max``/``min``/``prod``/``mean``/``any``/``all`` and the ``nan*`` forms) and the NumPy protocols
(``__array_ufunc__``, ``__array_function__``, ``@``), plus the fused ``sddmm`` and ``mttkrp`` example paths and the masked sparse product
``masked_matmul(s, a, b)`` = ``s * (a @ b)`` for sparse ``a``, ``b``.
Host code is Python; every data-path step is a hand-written CUDA kernel in ``libsparse_b200.so`` reached through a
thin C ABI (``include/sparse_b200.h``) via ctypes.  There is no CPU fallback: without the library or a CUDA device
operations raise.
"""
# the ufuncs / dtypes / constants of the Array-API namespace are NumPy's own objects: calling one on a sparse array goes
# through __array_ufunc__ to the device element-wise path (or raises TypeError if it is not in the CUDA op set)
from numpy import (add, bitwise_and, bitwise_not, bitwise_or, bitwise_xor, ceil, complex64, complex128, conj,  # noqa: F401
                   copysign, cos, cosh, divide, e, exp, expm1, finfo, float16, float32, float64, floor, floor_divide,
                   greater, greater_equal, hypot, iinfo, inf, int8, int16, int32, int64, isfinite, less, less_equal,
                   log, log1p, log2, log10, logaddexp, logical_and, logical_not, logical_or, logical_xor, maximum,
                   minimum, multiply, nan, negative, newaxis, nextafter, not_equal, pi, positive, reciprocal,
                   remainder, sign, signbit, sin, sinh, sqrt, square, subtract, tan, tanh, trunc, uint8, uint16,
                   uint32, uint64)
from numpy import arccos as acos  # noqa: F401
from numpy import arccosh as acosh  # noqa: F401
from numpy import arcsin as asin  # noqa: F401
from numpy import arcsinh as asinh  # noqa: F401
from numpy import arctan as atan  # noqa: F401
from numpy import arctan2 as atan2  # noqa: F401
from numpy import arctanh as atanh  # noqa: F401
from numpy import bool_ as bool  # noqa: F401
from numpy import invert as bitwise_invert  # noqa: F401
from numpy import left_shift as bitwise_left_shift  # noqa: F401
from numpy import power as pow  # noqa: F401
from numpy import right_shift as bitwise_right_shift  # noqa: F401

from ._argreduce import argmax, argmin
from ._settings import IS_NUMPY2 as _IS_NUMPY2
from ._coo import COO, as_coo
from ._creation import (abs, argwhere, asCOO, asarray, asnumpy, astype, broadcast_arrays, broadcast_shapes, can_cast, diff, empty, empty_like, equal, eye,
                        full, full_like, imag, interp, isinf, isnan, isneginf, isposinf, nonzero, ones, ones_like, real,
                        reshape, result_type, round, std, var, vecdot, zeros, zeros_like)
from ._dok import DOK
from ._dot import dot, matmul, tensordot
from ._einsum import einsum
from ._elemwise import broadcast_to, elemwise, where
from ._fused import masked_matmul, mttkrp, sddmm
from ._gcxs import CSC, CSR, GCXS
from ._io import load_npz, save_npz
from ._manip import (concatenate, diagonal, diagonalize, expand_dims, flip, kron, matrix_transpose, moveaxis, outer,
                     pad, permute_dims, repeat, roll, squeeze, stack, swapaxes, take, tile, tril, triu, unstack)
from ._nanreduce import nanmax, nanmean, nanmin, nanprod, nanreduce, nansum
from ._random import random
from ._sorting import sort, unique_counts, unique_values
from ._sparse_array import SparseArray

__version__ = "0.1.0"
# `__all__` below is exactly upstream's namespace (tests/test_namespace.py there); the fused example kernels `sddmm`,
# `mttkrp` and `masked_matmul`, the 2-D classes `CSR` / `CSC` and a few helpers are importable attributes outside of it.


def clip(a, min=None, max=None, out=None):
    """_coo/common.py:1028-1071."""
    return asCOO(a, name="clip").clip(min, max, out=out)


concat = concatenate


def sum(x, /, *, axis=None, dtype=None, keepdims=False):
    return x.sum(axis=axis, keepdims=keepdims, dtype=dtype)


def max(x, /, *, axis=None, keepdims=False):
    return x.max(axis=axis, keepdims=keepdims)


def min(x, /, *, axis=None, keepdims=False):
    return x.min(axis=axis, keepdims=keepdims)


def prod(x, /, *, axis=None, dtype=None, keepdims=False):
    return x.prod(axis=axis, keepdims=keepdims, dtype=dtype)


def mean(x, /, *, axis=None, keepdims=False, dtype=None):
    return x.mean(axis=axis, keepdims=keepdims, dtype=dtype)


def any(x, /, *, axis=None, keepdims=False):
    return x.any(axis=axis, keepdims=keepdims)


def all(x, /, *, axis=None, keepdims=False):
    return x.all(axis=axis, keepdims=keepdims)


__all__ = ["COO", "DOK", "GCXS", "SparseArray", "as_coo", "asarray", "tensordot", "matmul", "dot", "stack",
           "elemwise", "broadcast_to", "where", "random", "sum", "max", "min", "prod", "mean", "any", "all",
           "einsum", "save_npz", "load_npz", "nansum", "nanprod", "nanmean", "nanmax", "nanmin", "nanreduce",
           # array manipulation and creation next to the hot path (widened per SURVEY.md s8f)
           "concatenate", "concat", "unstack", "moveaxis", "permute_dims", "matrix_transpose", "squeeze",
           "expand_dims", "flip", "roll", "triu", "tril", "diagonal", "diagonalize", "pad", "repeat", "tile", "outer",
           "kron", "take", "clip", "eye", "full", "full_like", "zeros", "zeros_like", "ones", "ones_like", "empty",
           "empty_like", "asnumpy", "can_cast", "result_type", "std", "var", "abs", "reshape", "astype", "equal",
           "argmax", "argmin", "interp", "sort", "unique_values", "unique_counts", "round", "isinf", "isnan", "isposinf",
           "isneginf", "nonzero", "argwhere", "imag", "real", "vecdot", "diff", "asCOO", "broadcast_arrays",
           "broadcast_shapes",
           # NumPy's ufuncs, dtypes and constants under the Array-API names (sparse/numba_backend/__init__.py upstream)
           "acos", "acosh", "add", "asin", "asinh", "atan", "atan2", "atanh", "bitwise_and", "bitwise_invert",
           "bitwise_left_shift", "bitwise_not", "bitwise_or", "bitwise_right_shift", "bitwise_xor", "bool", "ceil",
           "complex128", "complex64", "conj", "copysign", "cos", "cosh", "divide", "e", "exp", "expm1", "finfo", "float16",
           "float32", "float64", "floor", "floor_divide", "greater", "greater_equal", "hypot", "iinfo", "inf", "int16",
           "int32", "int64", "int8", "isfinite", "less", "less_equal", "log", "log10", "log1p", "log2", "logaddexp",
           "logical_and", "logical_not", "logical_or", "logical_xor", "maximum", "minimum", "multiply", "nan", "negative",
           "newaxis", "nextafter", "not_equal", "pi", "positive", "pow", "reciprocal", "remainder", "sign", "signbit",
           "sin", "sinh", "sqrt", "square", "subtract", "tan", "tanh", "trunc", "uint16", "uint32", "uint64", "uint8"]

if _IS_NUMPY2:  # numpy.isdtype exists from NumPy 2.0 on (upstream adds it to the namespace under the same condition)
    from numpy import isdtype  # noqa: E402,F401

    __all__.append("isdtype")

__all__ = sorted(__all__)
