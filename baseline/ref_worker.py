#!/usr/bin/env python
"""Worker process of bench.py's CPU legs: times a CPU implementation of the C2 product on arrays the parent process
dumped as .npy files -- the same arrays the GPU arm multiplies.

    python baseline/ref_worker.py numba <dir> <steps> <warmup>
        The UNMODIFIED reference (oracle/_ref, installed by oracle/make_ref.sh): runs with PYTHONPATH=oracle/_ref so
        that `import sparse` is pydata/sparse's numba backend, in a process of its own (the product package never shares
        an interpreter with the reference).  The timed call is the reference's public API for the path,
        `sparse.tensordot(GCXS, ndarray, axes=1)` (numba_backend/_common.py:95 -> _dot :339 -> _dot_csr_ndarray
        :720-755): a `nopython, nogil` single-threaded kernel, so this is a 1-core number by construction.  Untimed
        warm-up calls absorb the numba JIT (as the reference's own harness does, examples/utils.py:15-16).
    python baseline/ref_worker.py port <dir> <steps> <warmup> <threads>
        The oracle's C restatement of the same loop (oracle/dot_oracle.c), OpenMP over rows with a FIXED thread count
        (the parent sets OMP_PROC_BIND=close OMP_PLACES=cores): the labelled "all cores" figure.

reads  <dir>/{a_data,a_indices,a_indptr,B}.npy + meta.json;  writes <dir>/C_<impl>.npy (last result), result_<impl>.json
"""
import json
import os
import sys
import time

import numpy as np


def main():
    impl, d, steps, warmup = sys.argv[1], sys.argv[2], int(sys.argv[3]), int(sys.argv[4])
    with open(os.path.join(d, "meta.json")) as f:
        meta = json.load(f)
    data = np.load(os.path.join(d, "a_data.npy"))
    indices = np.load(os.path.join(d, "a_indices.npy"))
    indptr = np.load(os.path.join(d, "a_indptr.npy"))
    B = np.load(os.path.join(d, "B.npy"))
    shape = tuple(meta["shape"])
    info = {}
    if impl == "numba":
        import numba
        import sparse  # the reference (PYTHONPATH=oracle/_ref)

        A = sparse.GCXS((data, indices, indptr), shape=shape, compressed_axes=(0,))

        def call():
            return sparse.tensordot(A, B, axes=1)

        info = {"sparse_version": sparse.__version__, "sparse_file": os.path.dirname(sparse.__file__),
                "numba": numba.__version__, "threads": 1,
                "api": "sparse.tensordot(GCXS, ndarray, axes=1) -> _dot_csr_ndarray (_common.py:720-755)"}
    elif impl == "port":
        sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
        import oracle

        threads = oracle.set_threads(int(sys.argv[5]))
        out_shape = (shape[0], B.shape[1])

        def call():
            return oracle.dot_csr_ndarray(out_shape, data, indices, indptr, B)

        info = {"threads": threads, "api": "oracle/dot_oracle.c orc_csr_dense (gcc -O3 -fopenmp, rows in parallel)",
                "omp_proc_bind": os.environ.get("OMP_PROC_BIND"), "omp_places": os.environ.get("OMP_PLACES")}
    else:
        raise SystemExit("ref_worker: unknown impl " + impl)
    for _ in range(max(warmup, 1)):
        C = call()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        C = call()
        ts.append(time.perf_counter() - t0)
    C = np.asarray(C)
    np.save(os.path.join(d, f"C_{impl}.npy"), C)
    info.update({"seconds": ts, "nnz": int(len(data)), "result_type": type(C).__name__, "result_dtype": str(C.dtype),
                 "host_cpus": os.cpu_count()})
    with open(os.path.join(d, f"result_{impl}.json"), "w") as f:
        json.dump(info, f)


if __name__ == "__main__":
    main()
