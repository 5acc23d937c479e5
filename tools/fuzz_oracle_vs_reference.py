#!/usr/bin/env python
"""Differential fuzzing of the ORACLE (oracle/dot_oracle.c, the CPU restatement the GPU parity tests compare with)
against the reference's own numba kernels; needs the reference installed in oracle/_ref (oracle/make_ref.sh).

    python tools/fuzz_oracle_vs_reference.py [--cases 400] [--seed 0]

The golden fixtures pin the oracle on 213 fixed kernel cases; this runs the same comparison on random ones: random
shapes (1..48, empty rows and columns, a fully dense product now and then), densities, every dtype pair the kernels
are specialised for (float32 / float64 / int32 / int64, mixed), REAL-valued data (so the summation order matters) with
exact zeros, cancellations (+x, -x pairs) and negative zeros mixed in.  Every output array is compared bit for bit:
dense results byte-wise, sparse results as (data, indices, indptr) / (coords, data) including the reference's
first-touch column order.  `_dot_csc_ndarray_sparse` reads an uninitialised tail upstream when sums cancel (DESIGN s4):
only the prefix both sides define is compared there.
"""
from __future__ import annotations

import argparse
import os
import sys
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
sys.path.insert(0, ROOT)

import sparse as R  # noqa: E402
from sparse.numba_backend import _common as C  # noqa: E402
from sparse.numba_backend import _umath as U  # noqa: E402
from sparse.numba_backend._coo import core as coo_core  # noqa: E402

import oracle as O  # noqa: E402

DTS = ["float32", "float64", "int32", "int64"]


def bits(x):
    x = np.ascontiguousarray(x)
    return x.view(np.uint8).reshape(-1) if x.size else np.empty(0, np.uint8)


def same(x, y):
    x, y = np.asarray(x), np.asarray(y)
    return x.shape == y.shape and x.dtype == y.dtype and np.array_equal(bits(x), bits(y))


def draw(rng, shape, dt, density):
    """Dense array with structure: zeros, +x/-x pairs (cancellation), a few -0.0."""
    dt = np.dtype(dt)
    mask = rng.random(shape) < density
    if dt.kind == "f":
        v = (rng.standard_normal(shape) * 3).astype(dt)
        v[rng.random(shape) < 0.15] = dt.type(1.5)
        v[rng.random(shape) < 0.15] = dt.type(-1.5)
        out = np.where(mask, v, dt.type(0))
        if out.size and rng.random() < 0.3:
            out.reshape(-1)[int(rng.integers(out.size))] = dt.type(-0.0)
    else:
        out = np.where(mask, rng.integers(-3, 4, size=shape), 0).astype(dt)
    return out


def csr(d):
    g = R.COO.from_numpy(d).asformat("gcxs", compressed_axes=(0,))
    return g.data, g.indices, np.asarray(g.indptr)


def csc(d):
    g = R.COO.from_numpy(d).asformat("gcxs", compressed_axes=(1,))
    return g.data, g.indices, np.asarray(g.indptr)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", type=int, default=400)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--max-extent", type=int, default=49, help="M, K, N are drawn below this (default 49)")
    args = ap.parse_args()
    O.build()
    bad, n = 0, 0
    counts = {}

    def check(name, i, ok, info):
        nonlocal bad, n
        n += 1
        counts[name] = counts.get(name, 0) + 1
        if not ok:
            bad += 1
            print(f"MISMATCH {name} case {i}: {info}", flush=True)

    warnings.simplefilter("ignore")
    for i in range(args.cases):
        rng = np.random.default_rng([args.seed, i])
        M, K, N = (int(v) for v in rng.integers(1, args.max_extent, size=3))
        if rng.random() < 0.1:
            M, K, N = (int(v) for v in rng.integers(1, 5, size=3))
        da_t, db_t = rng.choice(DTS), rng.choice(DTS)
        if rng.random() < 0.6:
            db_t = da_t
        dens_a = float(rng.choice([0.0, 0.05, 0.3, 0.7, 1.0]))
        dens_b = float(rng.choice([0.05, 0.3, 0.7, 1.0]))
        A, B = draw(rng, (M, K), da_t, dens_a), draw(rng, (K, N), db_t, dens_b)
        info = f"M={M} K={K} N={N} {da_t} x {db_t} dens {dens_a}/{dens_b} seed=({args.seed},{i})"
        out_shape = (M, N)
        ad, ai, ap_ = csr(A)
        cd, ci, cp = csc(A)
        bd, bi, bp = csr(B)
        a_coo, b_coo = R.COO.from_numpy(A), R.COO.from_numpy(B)
        # ---- csr @ dense (the headline kernel) and its sparse-output form
        want = C._dot_csr_ndarray_type(ad.dtype, B.dtype)(out_shape, ad, ai, ap_, B)
        check("csr_ndarray", i, same(O.dot_csr_ndarray(out_shape, ad, ai, ap_, B), want), info)
        wd, wi, wp = C._dot_csr_ndarray_type_sparse(ad.dtype, B.dtype)(out_shape, ad, ai, ap_, B)
        gd, gi, gp = O.dot_csr_ndarray_sparse(out_shape, ad, ai, ap_, B)
        check("csr_ndarray_sparse", i, same(gd, wd) and same(gi, wi) and same(gp, wp), info)
        # ---- csc @ dense
        want = C._dot_csc_ndarray_type(cd.dtype, B.dtype)((M, K), (K, N), cd, ci, cp, B)
        check("csc_ndarray", i, same(O.dot_csc_ndarray((M, K), (K, N), cd, ci, cp, B), want), info)
        wd, wi, wp = C._dot_csc_ndarray_type_sparse(cd.dtype, B.dtype)((M, K), (K, N), cd, ci, cp, B)
        gd, gi, gp, written = O.dot_csc_ndarray_sparse((M, K), (K, N), cd, ci, cp, B)
        # upstream counts structurally and fills numerically: entries past what it wrote are uninitialised memory.
        # Compare indptr, the sizes, and the prefix both sides define (the oracle reports how many entries it wrote).
        ok = (same(np.asarray(gp), np.asarray(wp)) and len(gd) == len(wd) and same(gd[:written], wd[:written])
              and same(gi[:written], np.asarray(wi[:written])))
        check("csc_ndarray_sparse(written prefix)", i, ok, info)
        # ---- csr @ csr (+ count) and coo @ coo
        check("csr_csr_count_nnz", i,
              int(O.csr_csr_count_nnz(out_shape, ai, bi, ap_, bp)) == int(C._csr_csr_count_nnz(out_shape, ai, bi, ap_, bp)),
              info)
        wd, wi, wp = C._dot_csr_csr_type(ad.dtype, bd.dtype)(out_shape, ad, bd, ai, bi, ap_, bp)
        gd, gi, gp = O.dot_csr_csr(out_shape, ad, bd, ai, bi, ap_, bp)
        check("csr_csr", i, same(gd, wd) and same(gi, wi) and same(np.asarray(gp), np.asarray(wp)), info)
        a_ip = np.concatenate([[0], np.cumsum(np.bincount(a_coo.coords[0], minlength=M))]).astype(np.intp)
        b_ip = np.concatenate([[0], np.cumsum(np.bincount(b_coo.coords[0], minlength=K))]).astype(np.intp)
        wc, wd = C._dot_coo_coo_type(a_coo.dtype, b_coo.dtype)(out_shape, a_coo.coords, b_coo.coords, a_coo.data,
                                                              b_coo.data, a_ip, b_ip)
        gc, gd = O.dot_coo_coo(out_shape, a_coo.coords, b_coo.coords, a_coo.data, b_coo.data, a_ip, b_ip)
        check("coo_coo", i, same(np.asarray(gc), np.asarray(wc)) and same(gd, wd), info)
        # ---- coo @ dense, dense @ coo (dense and sparse outputs)
        Bt = B.T
        want = C._dot_coo_ndarray_type(a_coo.dtype, Bt.dtype)(a_coo.coords, a_coo.data, Bt, out_shape)
        check("coo_ndarray", i, same(O.dot_coo_ndarray(a_coo.coords, a_coo.data, Bt, out_shape), want), info)
        wc, wd = C._dot_coo_ndarray_type_sparse(a_coo.dtype, Bt.dtype)(a_coo.coords, a_coo.data, Bt, out_shape)
        gc, gd = O.dot_coo_ndarray_sparse(a_coo.coords, a_coo.data, Bt, out_shape)
        check("coo_ndarray_sparse", i, same(np.asarray(gc).reshape(2, -1), np.asarray(wc).reshape(2, -1)) and same(gd, wd),
              info)
        want = C._dot_ndarray_coo_type(A.dtype, b_coo.dtype)(A, b_coo.coords, b_coo.data, out_shape)
        check("ndarray_coo", i, same(O.dot_ndarray_coo(A, b_coo.coords, b_coo.data, out_shape), want), info)
        bT = b_coo.T
        wc, wd = C._dot_ndarray_coo_type_sparse(A.dtype, bT.dtype)(A, bT.coords, bT.data, out_shape)
        gc, gd = O.dot_ndarray_coo_sparse(A, bT.coords, bT.data, out_shape)
        check("ndarray_coo_sparse", i, same(np.asarray(gc).reshape(2, -1), np.asarray(wc).reshape(2, -1)) and same(gd, wd),
              info)
        # ---- the element-wise matching helpers
        n1, n2, hi = int(rng.integers(0, 80)), int(rng.integers(0, 80)), int(rng.integers(1, 40))
        x = np.sort(rng.integers(0, hi, n1)).astype(np.intp)
        y = np.sort(rng.integers(0, hi, n2)).astype(np.intp)
        wa, wb = U._match_arrays(x, y)
        ga, gb = O.match_arrays(x, y)
        check("match_arrays", i, same(np.asarray(ga), np.asarray(wa)) and same(np.asarray(gb), np.asarray(wb)),
              f"n1={n1} n2={n2} hi={hi} seed=({args.seed},{i})")
        if n1:
            winv, wcnt = coo_core._calc_counts_invidx(x)
            ginv, gcnt = O.calc_counts_invidx(x)
            check("counts_invidx", i, same(np.asarray(ginv), np.asarray(winv)) and same(np.asarray(gcnt), np.asarray(wcnt)),
                  f"n1={n1} hi={hi} seed=({args.seed},{i})")
    print("comparisons per kernel:", ", ".join(f"{k} {v}" for k, v in counts.items()))
    print(f"TOTAL {n} comparisons over {args.cases} random cases, {bad} mismatches")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
