#!/usr/bin/env python
"""Masked sparse product `masked_matmul(s, a, b)` (K10) on seeded device-generated inputs; one JSON line per workload.

    python tools/bench_masked.py [--calls 10] [--warmup 2] [--only T1,T2,T3] [--cap-gb 30]

Workloads (inputs are generated on the device from a seed and are larger than the 126 MB L2):
  T1   symmetric ER-like graph, n = 1e6, average degree 32, f32 ones:       masked_matmul(A, A, A) and its .sum()
  T1s  the same model at n = 2.5e5, where the unfused expression fits comfortably (a like-for-like comparison)
  T2   symmetric Chung-Lu power-law graph, n = 1e6, nnz ~ 3.2e7, hubs of degree >= 1e4, f32 ones
  T3   distinct f64 operands: S 1e6 x 1e6 (nnz 1e7), A 1e6 x 1e5 (nnz 1e7), B 1e5 x 1e6 (nnz 1e7)

Reported per workload: the call time (ms, CUDA events, >= --calls calls after warm-up) of the public entry point and of
the K10 kernel alone; the intersection work sum over (i,j) in S of (|A_i| + |Bt_j|); a bytes model of the kernel (mask
in + values out + each A row once per non-empty mask row + Bt_j once per mask entry) over the kernel time, against
MEASURED_PEAKS.json's HBM bandwidth or else the data-sheet 7.7 TB/s (labelled); the unfused device path `s * (a @ b)`
where its estimated footprint is under --cap-gb (otherwise reported as skipped with the estimate); and parity: the
kernel's values on a seeded sample of mask rows bit-exact against the C restatement of upstream's product kernel
(oracle/, built by __graft_entry__.build()).  Writes nothing to the tree.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# bytes per product of the unfused path, as an estimate of its peak footprint: K4's upper-bound (index, value) layout,
# the pruned CSR product, and its COO form plus merge buffers in the element-wise multiply
BYTES_PER_PRODUCT = 40


def card():
    import torch

    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # the number is still reported, without its power limit
        pl = f"unknown ({type(e).__name__})"
    return name, pl


def peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 7700.0, "data sheet (HGX B200, 7.7 TB/s per GPU; not a measured figure)"


# ---- seeded inputs on the device ------------------------------------------------------------------------------------
def _csr(t, rows, cols, n_rows, vals):
    """CSR of entries already sorted by (row, column)."""
    indptr = t.zeros(n_rows + 1, dtype=t.int64, device=rows.device)
    indptr[1:] = t.cumsum(t.bincount(rows, minlength=n_rows), 0)
    return indptr, cols.contiguous(), vals.contiguous()


def _unique_edges(t, r, c, n_cols, symmetric):
    keep = r != c if symmetric else t.ones_like(r, dtype=t.bool)
    r, c = r[keep], c[keep]
    keys = t.cat([r * n_cols + c, c * n_cols + r]) if symmetric else r * n_cols + c
    keys = t.unique(keys)  # sorted, duplicates dropped
    return keys // n_cols, keys % n_cols


def er_graph(t, gen, n, deg):
    m = n * deg // 2
    r = t.randint(0, n, (m,), device="cuda", generator=gen)
    c = t.randint(0, n, (m,), device="cuda", generator=gen)
    rows, cols = _unique_edges(t, r, c, n, True)
    return _csr(t, rows, cols, n, t.ones(rows.numel(), dtype=t.float32, device="cuda"))


def chung_lu(t, gen, n, nnz, gamma=2.5, cap=50_000):
    w = t.arange(1, n + 1, device="cuda", dtype=t.float64).pow(-1.0 / (gamma - 1))
    w = w * (nnz / w.sum())
    w = w.clamp(max=cap)
    cdf = t.cumsum(w / w.sum(), 0)
    m = nnz // 2
    r = t.searchsorted(cdf, t.rand(m, device="cuda", dtype=t.float64, generator=gen)).clamp(max=n - 1)
    c = t.searchsorted(cdf, t.rand(m, device="cuda", dtype=t.float64, generator=gen)).clamp(max=n - 1)
    rows, cols = _unique_edges(t, r, c, n, True)
    return _csr(t, rows, cols, n, t.ones(rows.numel(), dtype=t.float32, device="cuda"))


def uniform(t, gen, shape, nnz, dtype):
    n_rows, n_cols = shape
    r = t.randint(0, n_rows, (nnz,), device="cuda", generator=gen)
    c = t.randint(0, n_cols, (nnz,), device="cuda", generator=gen)
    rows, cols = _unique_edges(t, r, c, n_cols, False)
    vals = (t.rand(rows.numel(), device="cuda", dtype=t.float64, generator=gen) * 2 - 1).to(dtype)
    return _csr(t, rows, cols, n_rows, vals)


# ---- measurement ----------------------------------------------------------------------------------------------------
def timed(t, fn, calls, warmup):
    for _ in range(warmup):
        fn()
    t.cuda.synchronize()
    e0, e1 = t.cuda.Event(enable_timing=True), t.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        out = fn()
    e1.record()
    t.cuda.synchronize()
    return e0.elapsed_time(e1) / calls, out


def oracle_rows(rows, s_csr, a_csr, b_csr, n_col):
    """s * (a @ b) at the stored positions of the sampled mask rows, from upstream's CSR @ CSR kernel restated in C."""
    import oracle

    (sp_, sc_, sv_), (ap_, ai_, av_), (bp_, bi_, bv_) = s_csr, a_csr, b_csr
    a_lens = ap_[rows + 1] - ap_[rows]
    a_ptr = np.concatenate([[0], np.cumsum(a_lens)])
    a_idx = np.concatenate([ai_[ap_[r]:ap_[r + 1]] for r in rows])
    a_val = np.concatenate([av_[ap_[r]:ap_[r + 1]] for r in rows])
    c_data, c_idx, c_ptr = oracle.dot_csr_csr((len(rows), n_col), a_val, bv_, a_idx, bi_, a_ptr, bp_)
    out = []
    for q, r in enumerate(rows):
        cols = sc_[sp_[r]:sp_[r + 1]]
        row_c = dict(zip(c_idx[c_ptr[q]:c_ptr[q + 1]].tolist(), c_data[c_ptr[q]:c_ptr[q + 1]]))
        acc = np.array([row_c.get(int(j), c_data.dtype.type(0)) for j in cols], dtype=c_data.dtype)
        acc = acc + c_data.dtype.type(0)
        out.append(sv_[sp_[r]:sp_[r + 1]] * acc.astype(sv_.dtype))
    return out


def run(name, S, A, B, shape, calls, warmup, cap_gb, with_sum):
    import torch as t

    import sparse_b200 as sp
    from sparse_b200 import _kernels as Kn
    from sparse_b200._gcxs import GCXS

    M, K = shape[0], shape[1]
    N = shape[2]
    s = GCXS._from_device(S[2], S[1], S[0], (M, N), (0,))
    a = GCXS._from_device(A[2], A[1], A[0], (M, K), (0,))
    b = GCXS._from_device(B[2], B[1], B[0], (K, N), (0,))
    nnz_s, nnz_a, nnz_b = int(S[1].numel()), int(A[1].numel()), int(B[1].numel())

    ms_call, res = timed(t, lambda: sp.masked_matmul(s, a, b), calls, warmup)
    ms_sum = None
    if with_sum:
        ms_sum, tot = timed(t, lambda: sp.masked_matmul(s, a, b).sum(), calls, warmup)

    # the kernel alone on the arrays the entry point hands it (int32 indices, Bt = b compressed by column)
    bcsc = b.change_compressed_axes((1,))
    bt_ptr, bt_idx, bt_val = bcsc._dev()[2], bcsc._dev()[1], bcsc._dev()[0]
    idx = [x.to(t.int32) for x in (S[0], S[1], A[0], A[1], bt_ptr, bt_idx)]
    ms_kernel, out = timed(t, lambda: Kn.masked_spgemm(idx[0], idx[1], S[2], idx[2], idx[3], A[2], idx[4], idx[5],
                                                        bt_val, M, N, K), calls, warmup)

    # counts from the shapes of the operands (computed on the device)
    s_rows = t.repeat_interleave(t.arange(M, device="cuda"), (S[0][1:] - S[0][:-1]))
    a_len = (A[0][1:] - A[0][:-1])
    bt_len = (bt_ptr[1:] - bt_ptr[:-1])
    work = int(a_len[s_rows].sum()) + int(bt_len[S[1]].sum())
    esz_v, esz_s, ib = A[2].element_size(), S[2].element_size(), 4
    touched = (S[0][1:] > S[0][:-1])
    bytes_model = (nnz_s * (ib + esz_s) + (M + 1) * ib            # mask in
                   + nnz_s * esz_s                                 # values out
                   + int(a_len[touched].sum()) * (ib + esz_v) + 2 * M * ib      # each A row once per mask row
                   + int(bt_len[S[1]].sum()) * (ib + esz_v) + 2 * nnz_s * ib)   # Bt_j once per mask entry
    gbs = bytes_model / (ms_kernel * 1e-3) / 1e9
    peak, peak_src = peak_gbs()

    # the unfused expression, when its estimated footprint fits under the cap
    b_len = (B[0][1:] - B[0][:-1])
    products = int(b_len[A[1]].sum())
    est_gb = products * BYTES_PER_PRODUCT / 1e9
    unfused = {"products": products, "estimated_gb": round(est_gb, 1), "cap_gb": cap_gb}
    if est_gb <= cap_gb:
        t.cuda.empty_cache()
        ms_unf, ures = timed(t, lambda: s * (a @ b), calls, 1)
        unfused.update(ms=round(ms_unf, 3), status="measured")
        # the fused result equals the unfused one at s's positions
        fc, uc = res.tocoo(), ures.tocoo()
        fk = fc.coords[0].astype(np.int64) * N + fc.coords[1]
        uk = uc.coords[0].astype(np.int64) * N + uc.coords[1]
        keep = np.isin(uk, fk)
        unfused["equal_at_s"] = bool(np.array_equal(fk, uk[keep]) and np.array_equal(
            fc.data.view(np.uint8), uc.data[keep].view(np.uint8)))
        del ures
    else:
        unfused["status"] = f"skipped: estimated {est_gb:.0f} GB > cap {cap_gb} GB"

    # parity on a seeded sample of mask rows
    rng = np.random.default_rng(0)
    nonempty = np.flatnonzero(touched.cpu().numpy())
    rows = np.sort(rng.choice(nonempty, size=min(256, len(nonempty)), replace=False))
    hub = int(t.argmax(S[0][1:] - S[0][:-1]))
    rows = np.unique(np.concatenate([rows, [hub]]))
    host = lambda arrs: tuple(x.cpu().numpy() for x in arrs)  # noqa: E731
    sh, ah = host(S), host(A)
    bh = host((B[0], B[1], B[2]))
    want = oracle_rows(rows, sh, ah, bh, N)
    got = out.cpu().numpy()
    parity = all(np.array_equal(got[sh[0][r]:sh[0][r + 1]].view(np.uint8), w.view(np.uint8))
                 for r, w in zip(rows, want))

    line = {"workload": name, "shape": [M, K, N], "nnz": {"s": nnz_s, "a": nnz_a, "b": nnz_b},
            "dtype": str(A[2].dtype).replace("torch.", ""), "calls": calls, "warmup": warmup,
            "ms_masked_matmul": round(ms_call, 3), "ms_kernel": round(ms_kernel, 3),
            "ms_masked_matmul_sum": None if ms_sum is None else round(ms_sum, 3),
            "result_nnz": int(res.nnz), "intersection_work": work, "bytes_model": bytes_model,
            "kernel_gbs_bytes_model": round(gbs, 1), "peak_gbs": peak, "peak_source": peak_src,
            "fraction_of_peak": round(gbs / peak, 4), "unfused": unfused,
            "parity_rows": int(len(rows)), "parity": bool(parity)}
    if with_sum:
        line["sum"] = float(np.asarray(tot.todense() if hasattr(tot, "todense") else tot)[()])
    return line


def main():
    p = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    p.add_argument("--calls", type=int, default=10)
    p.add_argument("--warmup", type=int, default=2)
    p.add_argument("--only", default="T1,T1s,T2,T3")
    p.add_argument("--cap-gb", type=float, default=30.0)
    args = p.parse_args()
    if args.calls < 10:
        p.error("--calls must be at least 10")
    import torch as t

    if not t.cuda.is_available():
        raise SystemExit("bench_masked.py needs a CUDA device (no CPU fallback)")
    from sparse_b200 import _lib

    _lib.load()
    name, power = card()
    gen = t.Generator(device="cuda")
    for w in args.only.split(","):
        gen.manual_seed({"T1": 1, "T1s": 11, "T2": 2, "T3": 3}[w])
        if w in ("T1", "T1s"):
            n = 1_000_000 if w == "T1" else 250_000
            A = er_graph(t, gen, n, 32)
            line = run(w, A, A, A, (n, n, n), args.calls, args.warmup, args.cap_gb, True)
        elif w == "T2":
            n = 1_000_000
            A = chung_lu(t, gen, n, 32_000_000)
            line = run(w, A, A, A, (n, n, n), args.calls, args.warmup, args.cap_gb, True)
            line["max_degree"] = int((A[0][1:] - A[0][:-1]).max())
        else:
            S = uniform(t, gen, (1_000_000, 1_000_000), 10_000_000, t.float64)
            A = uniform(t, gen, (1_000_000, 100_000), 10_000_000, t.float64)
            B = uniform(t, gen, (100_000, 1_000_000), 10_000_000, t.float64)
            line = run(w, S, A, B, (1_000_000, 100_000, 1_000_000), args.calls, args.warmup, args.cap_gb, False)
        line.update(gpu=name, power_limit=power)
        print(json.dumps(line), flush=True)
        del A
        t.cuda.empty_cache()


if __name__ == "__main__":
    main()
