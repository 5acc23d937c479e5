"""bench.py contract checks: the reference arm prints one well-formed JSON line and its --dump-outputs equal the
reference's own result (golden, tests/golden/make_bench_golden.py); on a GPU the dumped C equals the oracle's."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

SMALL = ["--rows", "4000", "--nnz", "80000", "--ncols", "128"]


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--rows", "4000",
                          "--nnz", "80000", "--ncols", "128", "--steps", "2", "--warmup", "1", "--cpu-rows", "2000"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "GNNZ/s" and line["value"] > 0
    cb = line["cpu_baseline"]
    if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "sparse", "__init__.py")):
        # the reference itself (numba, single-threaded by construction) + the labelled all-cores port figure
        assert cb["kind"] == "reference" and cb["cores"] == 1 and "numba" in cb and cb["value"] == line["value"]
        assert cb["all_cores_port"]["kind"] == "port" and cb["all_cores_port"]["cores"] >= 1
    else:  # oracle/_ref not installed (oracle/make_ref.sh): the C port stands in and says so
        assert cb["kind"] == "port" and cb["cores"] >= 1 and "oracle/_ref missing" in cb["sample"]
    assert "same arrays" in cb["sample"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]


def test_other_ranks_of_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--rows", "1000", "--nnz", "10000", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_reference_arm_dump_equals_the_references_result(tmp_path):
    """Inputs generated on the host (CUDA hidden): the same arrays on every machine, so the dumped C must be the one
    the reference's numba kernel computed for them, bit for bit -- whichever CPU implementation ran here."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "bench_reference_arm.npz"))
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", *SMALL, "--steps", "2",
                          "--warmup", "1", "--cpu-rows", "2000", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=300, cwd=ROOT,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 0, out.stderr[-2000:]
    C = np.load(tmp_path / "C.npy")
    rows = np.load(tmp_path / "C_rows.npy")
    assert C.dtype == np.float32 and rows.dtype == np.float64
    assert C.shape == tuple(g["shape"]) and np.array_equal(rows, np.arange(C.shape[0]))
    assert np.array_equal(C[g["rows"]].view(np.uint32), g["C_rows"].view(np.uint32))
    assert hashlib.sha256(C.tobytes()).hexdigest() == str(g["sha256"])


def test_dump_rows_fit_the_budget_and_do_not_change():
    M, ncols = 1_000_000, 128
    rows = bench.dump_rows(M, ncols)
    assert len(rows) * (ncols * 4 + 8) <= bench.DUMP_BYTES < (len(rows) + 1) * (ncols * 4 + 8)
    assert np.all(np.diff(rows) > 0) and rows[-1] < M
    assert np.array_equal(rows, bench.dump_rows(M, ncols))
    assert len(bench.dump_rows(M, ncols, share=4)) == len(rows) // 4
    assert np.array_equal(bench.dump_rows(1000, ncols), np.arange(1000))


@pytest.mark.gpu
def test_dump_outputs_equal_the_oracles_product(tmp_path):
    import torch

    import oracle

    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *SMALL, "--steps", "3", "--warmup", "1",
                          "--no-e2e", "--no-cpu", "--no-configs", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3
    dev = torch.device("cuda", 0)
    vals, cols, indptr, _ = bench.gen_A(torch, 4000, 4000, 80000, bench.A_SEED, dev)
    B = bench.gen_B(torch, 4000, 128, bench.B_SEED, dev)
    want = oracle.dot_csr_ndarray((4000, 128), vals.cpu().numpy(), cols.cpu().numpy().astype(np.int64),
                                  indptr.cpu().numpy().astype(np.int64), B.cpu().numpy())
    C = np.load(tmp_path / "C.npy")
    assert np.array_equal(np.load(tmp_path / "C_rows.npy"), np.arange(4000))
    assert np.array_equal(C.view(np.uint32), want.view(np.uint32))
