#!/usr/bin/env python
"""Golden output of bench.py's reference arm, computed by the reference itself (numba; installed into oracle/_ref by
oracle/make_ref.sh):

    python tests/golden/make_bench_golden.py

Runs `bench.py --impl reference` at the small size of tests/test_bench_contract.py with the inputs generated on the
host (CUDA hidden, so the seeded torch generators give the same arrays on every machine) and stores in
bench_reference_arm.npz the SHA-256 of the whole result C (float32 bytes) and a seeded sample of its rows.
"""
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
ARGS = ["--impl", "reference", "--rows", "4000", "--nnz", "80000", "--ncols", "128", "--steps", "2", "--warmup", "1",
        "--cpu-rows", "2000"]
SAMPLE_ROWS = 64


def main():
    with tempfile.TemporaryDirectory() as d:
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *ARGS, "--dump-outputs", d],
                             capture_output=True, text=True, check=True, cwd=ROOT,
                             env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["cpu_baseline"]["kind"] == "reference", "oracle/_ref is not installed (oracle/make_ref.sh)"
        C = np.load(os.path.join(d, "C.npy"))
        rows = np.load(os.path.join(d, "C_rows.npy"))
    assert np.array_equal(rows, np.arange(C.shape[0]))
    pick = np.sort(np.random.default_rng(0).choice(C.shape[0], SAMPLE_ROWS, replace=False))
    np.savez_compressed(os.path.join(HERE, "bench_reference_arm.npz"), shape=np.array(C.shape), rows=pick,
                        C_rows=C[pick], sha256=np.array(hashlib.sha256(C.tobytes()).hexdigest()))
    print("bench_reference_arm.npz:", C.shape, hashlib.sha256(C.tobytes()).hexdigest())


if __name__ == "__main__":
    main()
