#!/usr/bin/env python
"""Generate tests/golden/masked_spgemm_api.npz from the REFERENCE: upstream's unfused ``s * (a @ b)`` (and
``sum(a @ a * a)`` for the triangle cases), the expression ``masked_matmul`` computes without forming ``a @ b``.

Run in the authoring container only (needs the pydata/sparse checkout and numba):

    python tests/golden/make_masked_golden.py

Like make_golden.py, the reference is imported from a scratch copy under a temp dir; nothing from its sources is
copied into the repo.  Operands are stored as canonical COO (the test converts them to the case's format), except
operands with unsorted rows, which are stored as the raw GCXS arrays an earlier ``GCXS @ GCXS`` produced.  For each
case the full upstream result is stored (``out_``) together with that result restricted to the stored positions of
`s` (``r_``), and ``outright`` says whether the two are the same.
"""
from __future__ import annotations

import json
import os
import shutil
import sys
import tempfile
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("SPARSE_REFERENCE", "/root/reference")


def import_reference():
    tmp = os.path.join(tempfile.gettempdir(), "sparse_b200_refcopy_masked")
    if os.path.isdir(tmp):
        shutil.rmtree(tmp)
    shutil.copytree(os.path.join(REF, "sparse"), os.path.join(tmp, "sparse"))
    with open(os.path.join(tmp, "sparse", "_version.py"), "w") as f:
        f.write('__version__ = "0.0.0+ref"\n__version_tuple__ = (0, 0, 0)\n')
    sys.path.insert(0, tmp)
    import sparse  # noqa: E402

    assert sparse.__file__.startswith(tmp)
    return sparse


sparse = import_reference()

FORMATS = {"coo": ("coo", None), "csr": ("gcxs", (0,)), "csc": ("gcxs", (1,))}


def enc(prefix, x):
    out = {}
    if isinstance(x, sparse.COO):
        out[prefix + "kind"] = "coo"
        out[prefix + "coords"] = x.coords
        out[prefix + "data"] = x.data
    else:
        out[prefix + "kind"] = "gcxs"
        out[prefix + "data"] = x.data
        out[prefix + "indices"] = x.indices
        out[prefix + "indptr"] = np.asarray(x.indptr)
        out[prefix + "ca"] = np.array(x.compressed_axes, dtype=np.int64)
    out[prefix + "shape"] = np.array(x.shape, dtype=np.int64)
    out[prefix + "fill"] = np.asarray(x.fill_value)
    return out


def enc_operand(prefix, x):
    """Canonical COO of `x`, or the raw arrays of a GCXS whose rows are stored unsorted."""
    if isinstance(x, sparse.GCXS) and not all(
            (np.diff(x.indices[x.indptr[r]:x.indptr[r + 1]]) > 0).all() for r in range(len(x.indptr) - 1)):
        return enc(prefix, x)
    return enc(prefix, sparse.COO(x.tocoo() if isinstance(x, sparse.GCXS) else x))


def as_fmt(x, fmt):
    kind, ca = FORMATS[fmt]
    return x.asformat("coo") if kind == "coo" else x.asformat("gcxs", compressed_axes=ca)


def rand(rng, shape, density, dtype, values="small"):
    """Random COO; values: "small" = small signed integers (exact cancellations), "real" = floats in [-1, 1)."""
    n = int(round(density * shape[0] * shape[1])) if shape[0] * shape[1] else 0
    lin = np.unique(rng.integers(0, max(shape[0] * shape[1], 1), size=n)) if n else np.zeros(0, np.int64)
    coords = np.stack([lin // max(shape[1], 1), lin % max(shape[1], 1)]) if n else np.zeros((2, 0), np.int64)
    dt = np.dtype(dtype)
    if dt == np.bool_:
        data = np.ones(len(lin), dtype=bool)
    elif values == "small":
        data = rng.choice(np.array([-3, -2, -1, 1, 2, 3]), size=len(lin)).astype(dt)
    elif values == "wrap":
        data = rng.integers(-120, 120, size=len(lin)).astype(dt)
        data[data == 0] = 7
    elif values == "big":  # products and sums that wrap in 32 (and, for 64-bit types, 64) bits
        hi = 2**40 if dt.itemsize == 8 else 60_000
        data = rng.integers(1, hi, size=len(lin)).astype(dt)
    else:
        data = (rng.random(len(lin)) * 2 - 1).astype(dt)
    return sparse.COO(coords, data, shape=shape, has_duplicates=False, sorted=True)


class Book:
    def __init__(self):
        self.arrays, self.cases = {}, []

    def add(self, info, s, a, b, triangles=False):
        with np.errstate(all="ignore"):
            out = s * (a @ b)
        sc = sparse.COO(s.tocoo() if isinstance(s, sparse.GCXS) else s)
        oc = sparse.COO(out.tocoo() if isinstance(out, sparse.GCXS) else out)
        skeys = sc.coords[0] * s.shape[1] + sc.coords[1]
        okeys = oc.coords[0] * s.shape[1] + oc.coords[1]
        keep = np.isin(okeys, skeys)
        r = sparse.COO(oc.coords[:, keep], oc.data[keep], shape=oc.shape, has_duplicates=False, sorted=True,
                       fill_value=oc.fill_value)
        if isinstance(out, sparse.GCXS):
            r = r.asformat("gcxs", compressed_axes=out.compressed_axes)
        i = len(self.cases)
        info = dict(info, outright=bool(keep.all()))
        if triangles:
            with np.errstate(all="ignore"):
                tri = (a @ a * a).sum()
                info["triangles"] = repr(np.asarray(tri.todense() if hasattr(tri, "todense") else tri)[()].item())
        self.cases.append(info)
        arrs = {**enc_operand("s_", s), **enc_operand("a_", a), **enc_operand("b_", b), **enc("out_", out),
                **enc("r_", r)}
        for k, v in arrs.items():
            self.arrays[f"c{i}__{k}"] = np.asarray(v)

    def save(self):
        self.arrays["meta"] = np.array(json.dumps(self.cases))
        path = os.path.join(HERE, "masked_spgemm_api.npz")
        np.savez_compressed(path, **self.arrays)
        print(f"{path}: {len(self.cases)} cases, {os.path.getsize(path)} bytes")


def main():
    bk = Book()
    rng = np.random.default_rng(20261017)
    M, K, N = 9, 11, 10

    # every format triple of s / a / b, float64 with exact cancellations (to +0 and, times a negative s, to -0)
    for fs in FORMATS:
        for fa in FORMATS:
            for fb in FORMATS:
                s, a, b = rand(rng, (M, N), 0.5, "f8"), rand(rng, (M, K), 0.4, "f8"), rand(rng, (K, N), 0.4, "f8")
                bk.add(dict(name=f"fmt-{fs}-{fa}-{fb}", fs=fs, fa=fa, fb=fb), as_fmt(s, fs), as_fmt(a, fa),
                       as_fmt(b, fb))

    # dtypes (s, a, b); real-valued floats make the summation order visible in the last bits
    dtypes = [("f4", "f4", "f4", "real"), ("f8", "f8", "f8", "real"), ("i4", "i4", "i4", "small"),
              ("i8", "i8", "i8", "small"), ("?", "?", "?", "small"), ("i1", "i1", "i1", "wrap"),
              ("f4", "i8", "f4", "real"), ("f4", "f4", "f8", "real"), ("?", "?", "i8", "small"),
              ("i8", "?", "?", "small"), ("f8", "i8", "i8", "small"), ("f4", "?", "?", "small")]
    for ds, da, db, vals in dtypes:
        for fmt in ("coo", "csr", "csc"):
            s, a, b = (rand(rng, (M, N), 0.5, ds, vals), rand(rng, (M, K), 0.5, da, vals),
                       rand(rng, (K, N), 0.5, db, vals))
            bk.add(dict(name=f"dtype-{ds}-{da}-{db}-{fmt}", fs=fmt, fa=fmt, fb=fmt), as_fmt(s, fmt), as_fmt(a, fmt),
                   as_fmt(b, fmt))

    # NaN / inf inside s, and inside a / b on products that land in s
    for where in ("s", "ab"):
        for fmt in ("coo", "csr"):
            s, a, b = rand(rng, (M, N), 0.6, "f8"), rand(rng, (M, K), 0.5, "f8"), rand(rng, (K, N), 0.5, "f8")
            x = s if where == "s" else a
            d = x.data.copy()
            d[::4] = np.inf
            d[1::5] = np.nan
            d[2::7] = -np.inf
            x = sparse.COO(x.coords, d, shape=x.shape, has_duplicates=False, sorted=True)
            s, a = (x, a) if where == "s" else (s, x)
            bk.add(dict(name=f"nonfinite-{where}-{fmt}", fs=fmt, fa=fmt, fb=fmt), as_fmt(s, fmt), as_fmt(a, fmt),
                   as_fmt(b, fmt))

    # empty rows, an empty mask, zero-length axes
    s, a, b = rand(rng, (M, N), 0.5, "f8"), rand(rng, (M, K), 0.5, "f8"), rand(rng, (K, N), 0.5, "f8")
    keep_a = a.coords[0] % 3 != 1
    a = sparse.COO(a.coords[:, keep_a], a.data[keep_a], shape=a.shape)
    keep_s = s.coords[0] % 4 != 2
    s = sparse.COO(s.coords[:, keep_s], s.data[keep_s], shape=s.shape)
    for fmt in ("coo", "csr", "csc"):
        bk.add(dict(name=f"empty-rows-{fmt}", fs=fmt, fa=fmt, fb=fmt), as_fmt(s, fmt), as_fmt(a, fmt), as_fmt(b, fmt))
        bk.add(dict(name=f"empty-mask-{fmt}", fs=fmt, fa=fmt, fb=fmt), as_fmt(rand(rng, (M, N), 0.0, "f8"), fmt),
               as_fmt(a, fmt), as_fmt(b, fmt))
    for (m, k, n) in ((0, K, N), (M, 0, N), (M, K, 0)):
        for fmt in ("coo", "csr"):
            if fmt == "csr" and 0 in (m, k, n):
                fmts = ("coo", "coo", "coo") if (m == 0 or n == 0) else ("csr", "csr", "csr")
            else:
                fmts = (fmt, fmt, fmt)
            s, a, b = rand(rng, (m, n), 0.5, "f8"), rand(rng, (m, k), 0.5, "f8"), rand(rng, (k, n), 0.5, "f8")
            bk.add(dict(name=f"zero-axis-{m}x{k}x{n}-{fmts[0]}", fs=fmts[0], fa=fmts[1], fb=fmts[2]),
                   as_fmt(s, fmts[0]), as_fmt(a, fmts[1]), as_fmt(b, fmts[2]))

    # triangles: symmetric 0/1 adjacency, the mask equal to a
    for dt in ("f8", "i8", "f4"):
        x = rand(rng, (40, 40), 0.15, dt)
        x = sparse.COO(x.coords, np.ones(x.nnz, dtype=dt), shape=x.shape)
        x = ((x + x.T) != 0).astype(dt)
        x = sparse.COO(x.coords[:, x.coords[0] != x.coords[1]], x.data[x.coords[0] != x.coords[1]], shape=x.shape)
        for fmt in ("coo", "csr"):
            g = as_fmt(x, fmt)
            bk.add(dict(name=f"triangles-{dt}-{fmt}", fs=fmt, fa=fmt, fb=fmt), g, g, g, triangles=True)

    # rows longer than the kernel's shared-memory stage (512 entries), and a hub mask row with many entries
    a = rand(rng, (4, 1500), 0.05, "f8", "real")
    hub = sparse.COO(np.stack([np.zeros(900, np.int64), np.sort(rng.choice(1500, 900, replace=False))]),
                     rng.random(900) * 2 - 1, shape=(4, 1500))
    a = sparse.COO(np.concatenate([a.coords[:, a.coords[0] != 0], hub.coords], axis=1),
                   np.concatenate([a.data[a.coords[0] != 0], hub.data]), shape=(4, 1500))
    b = rand(rng, (1500, 200), 0.015, "f8", "real")
    s = rand(rng, (4, 200), 0.2, "f8", "real")
    s = sparse.COO(np.concatenate([s.coords[:, s.coords[0] != 1], np.stack([np.ones(200, np.int64), np.arange(200)])],
                                  axis=1), np.concatenate([s.data[s.coords[0] != 1], rng.random(200) + 0.5]),
                   shape=(4, 200))
    for fmt in ("coo", "csr"):
        bk.add(dict(name=f"long-rows-{fmt}", fs=fmt, fa=fmt, fb=fmt), as_fmt(s, fmt), as_fmt(a, fmt), as_fmt(b, fmt))

    # operands with unsorted rows: results of an earlier GCXS @ GCXS (reverse first-touch column order per row)
    for dt in ("f8", "f4", "i8"):
        for ca in ((0,), (1,)):
            vals = "real" if dt != "i8" else "small"
            x = rand(rng, (M, 6), 0.5, dt, vals).asformat("gcxs", compressed_axes=ca)
            y = rand(rng, (6, K), 0.5, dt, vals).asformat("gcxs", compressed_axes=ca)
            z = rand(rng, (K, 5), 0.5, dt, vals).asformat("gcxs", compressed_axes=ca)
            w = rand(rng, (5, N), 0.5, dt, vals).asformat("gcxs", compressed_axes=ca)
            a, b = x @ y, z @ w
            s = as_fmt(rand(rng, (M, N), 0.6, dt, vals), "csr" if ca == (0,) else "csc")
            fa = fb = "raw"
            bk.add(dict(name=f"unsorted-{dt}-ca{ca[0]}", fs="csr" if ca == (0,) else "csc", fa=fa, fb=fb), s, a, b)
            bk.add(dict(name=f"unsorted-{dt}-ca{ca[0]}-coo-mask", fs="coo", fa=fa, fb=fb), sparse.COO(s.tocoo()), a, b)

    # integer products (narrow, unsigned, wrapping) under a floating-point mask: upstream's product wraps in its own
    # integer dtype before the multiply by s promotes it
    for ds, dab, vals in (("f4", "i4", "big"), ("f8", "i4", "big"), ("f8", "u1", "wrap"), ("f8", "i2", "wrap"),
                          ("f4", "i1", "wrap"), ("f4", "u2", "wrap"), ("f8", "u8", "big"), ("f8", "u4", "big")):
        for fmt in ("coo", "csr", "csc"):
            s = rand(rng, (M, N), 0.5, ds, "real")
            a, b = rand(rng, (M, K), 0.5, dab, vals), rand(rng, (K, N), 0.5, dab, vals)
            bk.add(dict(name=f"intfloat-{ds}-{dab}-{fmt}", fs=fmt, fa=fmt, fb=fmt), as_fmt(s, fmt), as_fmt(a, fmt),
                   as_fmt(b, fmt))
    for ds, dab in (("f8", "i2"), ("f4", "u1")):  # zero-length contraction: upstream's product is an empty COO
        s = rand(rng, (M, N), 0.5, ds, "real")
        a, b = rand(rng, (M, 0), 0.5, dab, "wrap"), rand(rng, (0, N), 0.5, dab, "wrap")
        bk.add(dict(name=f"intfloat-zero-k-{ds}-{dab}", fs="csr", fa="csr", fb="csr"), as_fmt(s, "csr"),
               as_fmt(a, "csr"), as_fmt(b, "csr"))
    bk.save()


if __name__ == "__main__":
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        main()
