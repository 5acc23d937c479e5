#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (BASELINE.json: configs[1] = C2).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--gather ce|nccl] [--dump-outputs DIR]

Workload C2: GCXS/CSR A (1e6 x 1e6, nnz 1e8, fp32, uniform-random positions) times dense
B (1e6 x 128 fp32) -> dense C, i.e. ``sparse.tensordot(A, B, axes=1)`` -> _dot_csr_ndarray
(reference: sparse/numba_backend/_common.py:720-755).  A "step" is one full product.

* ``value``    GNNZ/s, device-resident inputs, CUDA-event timed, max over ranks.
* ``e2e``      the same product through the host-buffer C-ABI call (b2s_spmm_csr_dense_host):
               pinned host arrays in, host array out, H2D/D2H inside the timed region.
* ``roofline`` algorithmic bytes (gather model, SURVEY.md s8(d): 525 B/nnz with int32 indices)
               / measured kernel time, against MEASURED_PEAKS.json's HBM copy bandwidth.
* ``cpu_baseline``  the REFERENCE ITSELF -- pydata/sparse's numba path (oracle/_ref, oracle/make_ref.sh), called as
               sparse.tensordot(GCXS, ndarray, axes=1) in a worker process (baseline/ref_worker.py), 1 core (the
               kernel is single-threaded by construction) -- on the first 1e5 rows of the very arrays the GPU
               multiplies, its output bit-compared with the GPU's rows; plus a labelled all-cores figure from the
               OpenMP port (oracle/dot_oracle.c, fixed 32 threads, OMP_PROC_BIND=close).
* ``configs``  the other BASELINE.json configs (C1, C3, C3-large, C4, C5, reductions, MTTKRP): ms, roofline
               fraction by the SURVEY s8(d) formula, parity against the oracle (tools/bench_configs.py); N = 1 only.
* N > 1: ``value`` is WEAK scaling -- every rank owns a 1e6-row block of A (nnz 1e8) and a K/N row shard of B;
  each step gathers B (copy engines over NVLink: sparse_b200._dist.PeerGather; --gather nccl = the NCCL
  all-gather) and runs K1 on the local row block.  ``strong`` = the named 1e8-nnz problem cut into nnz-balanced row
  blocks over the N GPUs, with B replicated (no collective) and with B row-sharded (gather every step).

Inputs are synthetic (seeded torch generators on the device); 2.2 GB of operands per rank is far
larger than the 126 MB L2, so no explicit L2 flush is needed between steps ("l2": "inputs>L2").

``--dump-outputs DIR`` writes what the timed path returned in its last step: ``C.npy`` (float32) holds rows of C and
``C_rows.npy`` (float64) their row indices -- all rows when C fits in 64 MB, else a fixed seeded sample of rows.  With
the same arguments the inputs are the same on every run, so two builds can be compared output for output.  With N > 1
(weak scaling: every rank multiplies its OWN M-row matrix A, seeded A_SEED + rank) every rank writes ``C_rank<r>.npy``
/ ``C_rows_rank<r>.npy`` for its own product, within 64 MB / N; the row indices are local to that product, so the files
are N separate results, not blocks of one C.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--rows", type=int, default=1_000_000, help="M (= K) of the C2 workload")
    p.add_argument("--nnz", type=int, default=100_000_000)
    p.add_argument("--ncols", type=int, default=128)
    p.add_argument("--variant", type=int, default=0, help="K1 variant override (1 LDG dynamic rows = default, 2 bulk-TMA, 3 LDG static grid)")
    p.add_argument("--unroll", type=int, default=0)
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-cpu", action="store_true")
    p.add_argument("--cpu-rows", type=int, default=0, help="rows of A in the CPU-baseline sample (0 = auto)")
    p.add_argument("--gather", default="ce", choices=["ce", "nccl"], help="N>1: transport of the per-step gather of B")
    p.add_argument("--no-strong", action="store_true", help="N>1: skip the strong-scaling block")
    p.add_argument("--no-configs", action="store_true", help="N=1: skip the per-config block (C1, C3, C4, C5, ...)")
    p.add_argument("--no-numa", action="store_true", help="do not pin the process to the GPU's NUMA node")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write C of the last timed step (or a seeded row sample of it, 64 MB at most) as .npy files")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    return args


# ----------------------------------------------------------------------------------------------
def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def known_traffic(ncols):
    """Per-launch DRAM bytes of K1 from the committed ncu --set full capture (profiles/), if any."""
    path = os.path.join(ROOT, "profiles", "k1_traffic.json")
    try:
        with open(path) as f:
            d = json.load(f)
        if int(d.get("ncols", 128)) == ncols:
            return float(d["dram_bytes_per_launch"])
    except Exception:
        pass
    return None


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.samples = []
        self.stamps = []
        self.window = None  # (t0, t1) wall-clock bounds of the timed region, set by the caller
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        # one nvidia-smi process in loop mode (-lms 20): dense samples even for a timed region of ~100 ms
        try:
            self._proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index),
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self._proc.stdout:
                line = line.strip()
                if line:
                    self.samples.append([x.strip() for x in line.split(",")])
                    self.stamps.append(time.time())
                if self._stop.is_set():
                    break
        except Exception:
            pass

    def __enter__(self):
        self._proc = None
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        time.sleep(0.15)  # let the sampler start before the timed region
        return self

    def __exit__(self, *a):
        time.sleep(0.05)
        self._stop.set()
        if self._proc is not None:
            try:
                self._proc.terminate()
            except Exception:
                pass
        self._t.join(timeout=3)

    def summary(self):
        if self.window is not None and self.samples:
            t0, t1 = self.window
            inside = [s for s, t in zip(self.samples, self.stamps) if t0 - 0.02 <= t <= t1 + 0.02]
            # a region shorter than the sampling period: take the samples nearest to it
            if not inside:
                order = sorted(range(len(self.samples)), key=lambda i: abs(self.stamps[i] - 0.5 * (t0 + t1)))
                inside = [self.samples[i] for i in order[:3]]
            self.samples = inside
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[3 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples)}


# ----------------------------------------------------------------------------------------------
A_SEED, B_SEED = 1234, 4321  # A is seeded per rank (A_SEED + rank); B is ONE matrix for the whole job


def gen_A(torch, M, K, nnz, seed, device):
    """Uniform-random CSR (sorted unique columns per row), generated on `device`: vals f32, cols i32, indptr i32."""
    g = torch.Generator(device=device).manual_seed(seed)
    lin = torch.randint(0, M * K, (int(nnz * 1.0006) + 1024,), generator=g, device=device, dtype=torch.int64)
    lin = torch.unique(lin)  # sorted
    extra = lin.numel() - nnz
    if extra > 0:  # drop `extra` entries at random positions -> exactly nnz
        keep = torch.ones(lin.numel(), dtype=torch.bool, device=device)
        while extra > 0:
            idx = torch.randint(0, lin.numel(), (extra,), generator=g, device=device)
            keep[idx] = False
            extra = int(keep.sum().item()) - nnz
            if extra < 0:  # dropped too many duplicates impossible; re-add is not needed
                break
        lin = lin[keep]
    rows = torch.div(lin, K, rounding_mode="floor")
    cols = (lin - rows * K).to(torch.int32)
    counts = torch.bincount(rows, minlength=M)
    indptr = torch.zeros(M + 1, dtype=torch.int64, device=device)
    indptr[1:] = torch.cumsum(counts, 0)
    del lin, rows, counts
    vals = torch.rand(cols.numel(), generator=g, device=device, dtype=torch.float32)
    return vals, cols, indptr.to(torch.int32), g


def gen_B(torch, K, ncols, seed, device):
    g = torch.Generator(device=device).manual_seed(seed)
    return torch.rand((K, ncols), generator=g, device=device, dtype=torch.float32)


def make_workload(torch, M, K, nnz, ncols, seed, device, b_seed=None):
    """A (gen_A) + dense B.  b_seed=None draws B from A's generator (tools/ and tests use this form); the bench
    passes b_seed so that every rank of a job holds the same B."""
    vals, cols, indptr, g = gen_A(torch, M, K, nnz, seed, device)
    if b_seed is None:
        B = torch.rand((K, ncols), generator=g, device=device, dtype=torch.float32)
    else:
        B = gen_B(torch, K, ncols, b_seed, device)
    return vals, cols, indptr, B


def algorithmic_bytes(nnz, M, ncols, vb=4, ib=4):
    """SURVEY.md s8(d) gather model: A stream + indptr + one B row per nnz + C written once."""
    return nnz * (vb + ib) + (M + 1) * ib + nnz * ncols * vb + M * ncols * vb


DUMP_BYTES = 64_000_000  # --dump-outputs: payload of all files together (the .npy headers fit in the slack)
DUMP_SEED = 2024


def dump_rows(M, ncols, share=1):
    """Rows of an M x ncols fp32 C that --dump-outputs writes: all of them when they fit in DUMP_BYTES / share, else a
    fixed seeded sample (sorted), the same on every run.  Each row costs ncols * 4 bytes of C + 8 for its index."""
    n = DUMP_BYTES // share // (ncols * 4 + 8)
    if M <= n:
        return np.arange(M)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(M, size=n, replace=False))


def write_outputs(d, c_rows, rows, suffix=""):
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, f"C{suffix}.npy"), np.ascontiguousarray(c_rows, dtype=np.float32))
    np.save(os.path.join(d, f"C_rows{suffix}.npy"), rows.astype(np.float64))


# ---- CPU legs: the reference (numba) and the OpenMP port, each in a worker process, on dumped arrays -------------------
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
WORKER = os.path.join(ROOT, "baseline", "ref_worker.py")
CPU_ROWS = 100_000      # rows of A in the CPU sample (x full B): ~1e7 nnz, ~0.5 s per numba call
PORT_THREADS = 32       # fixed; does not follow OMP_NUM_THREADS (torchrun exports 1)


def have_reference():
    return os.path.exists(os.path.join(REF_DIR, "sparse", "__init__.py"))


def dump_sample(vals, cols, indptr, B, rows_sample, K):
    """Write the first `rows_sample` rows of A (int64 indices, the reference's own layout) and the full B as .npy."""
    import tempfile

    need = int(B.numel()) * 4 * 2 + (64 << 20)  # B + the sample of A + the results, with slack
    base = None
    try:
        st = os.statvfs("/dev/shm")
        if os.access("/dev/shm", os.W_OK) and st.f_bavail * st.f_frsize > need + int(indptr[rows_sample].item()) * 24:
            base = "/dev/shm"
    except OSError:
        pass
    d = tempfile.mkdtemp(prefix="b2s_ref_", dir=base)
    ip = indptr[: rows_sample + 1].cpu().numpy().astype(np.int64)
    n = int(ip[-1])
    np.save(os.path.join(d, "a_data.npy"), vals[:n].cpu().numpy())
    np.save(os.path.join(d, "a_indices.npy"), cols[:n].cpu().numpy().astype(np.int64))
    np.save(os.path.join(d, "a_indptr.npy"), ip)
    np.save(os.path.join(d, "B.npy"), B.cpu().numpy())
    with open(os.path.join(d, "meta.json"), "w") as f:
        json.dump({"op": "csr_dense", "shape": [rows_sample, K]}, f)
    return d, n


def run_worker(impl, d, steps, warmup, threads=None, timeout=900):
    env = {k: v for k, v in os.environ.items() if not k.startswith(("OMP_", "NUMBA_", "MKL_"))}
    cmd = [sys.executable, WORKER, impl, d, str(steps), str(warmup)]
    if impl == "numba":
        env["PYTHONPATH"] = REF_DIR
        env["NUMBA_CACHE_DIR"] = os.path.join(d, "numba_cache")
    else:
        env.update({"OMP_NUM_THREADS": str(threads), "OMP_PROC_BIND": "close", "OMP_PLACES": "cores"})
        env.pop("PYTHONPATH", None)
        cmd.append(str(threads))
    r = subprocess.run(cmd, env=env, cwd=d, capture_output=True, text=True, timeout=timeout)
    if r.returncode != 0:
        raise RuntimeError(f"ref_worker {impl} failed: {r.stderr[-2000:]}")
    with open(os.path.join(d, f"result_{impl}.json")) as f:
        return json.load(f)


def cpu_legs(vals, cols, indptr, B, K, ncols, rows_sample, steps, warmup, gpu_rows=None, dump_dir=None):
    """Time the reference (numba, 1 core) and the port (fixed threads) on the same dumped sample.  Returns the
    `cpu_baseline` object; when `gpu_rows` (the GPU's C[:rows_sample] as a host array) is given, both outputs are
    bit-compared with it.  `dump_dir`: write the last result of the reference (of the port when the reference is not
    installed) there, as --dump-outputs does."""
    import shutil

    d, n = dump_sample(vals, cols, indptr, B, rows_sample, K)
    sample = (f"first {rows_sample} rows of the GPU arm's own A ({n} nnz, int64 indices) x the full B({K}x{ncols}), "
              f"same arrays (dumped as .npy)")
    try:
        out = {}
        if have_reference():
            r = run_worker("numba", d, steps, warmup)
            best, med = min(r["seconds"]), float(np.median(r["seconds"]))
            out = {"value": round(n / med / 1e9, 5), "unit": "GNNZ/s", "cores": 1, "kind": "reference",
                   "sample": sample + f"; {steps} timed calls after {max(warmup, 1)} warm-up (JIT), median",
                   "best": round(n / best / 1e9, 5), "api": r["api"], "numba": r["numba"],
                   "host_cpus": r["host_cpus"]}
            if gpu_rows is not None:
                c = np.load(os.path.join(d, "C_numba.npy"))
                out["parity_bit_exact_vs_gpu"] = bool(c.shape == gpu_rows.shape and np.array_equal(
                    c.view(np.uint32), gpu_rows.view(np.uint32)))
        threads = min(PORT_THREADS, os.cpu_count() or 1)
        r = run_worker("port", d, steps, max(warmup, 1), threads=threads)
        med = float(np.median(r["seconds"]))
        port = {"value": round(n / med / 1e9, 5), "unit": "GNNZ/s", "cores": r["threads"], "kind": "port",
                "best": round(n / min(r["seconds"]) / 1e9, 5),
                "note": "oracle/dot_oracle.c, OpenMP over rows, OMP_PROC_BIND=close OMP_PLACES=cores, same sample"}
        if gpu_rows is not None:
            c = np.load(os.path.join(d, "C_port.npy"))
            port["parity_bit_exact_vs_gpu"] = bool(np.array_equal(c.view(np.uint32), gpu_rows.view(np.uint32)))
        if out:
            out["all_cores_port"] = port
        else:  # oracle/_ref is not installed: the port is all there is (and says so)
            out = dict(port, sample=sample + "; oracle/_ref missing (see oracle/make_ref.sh), so this is the C port")
        if dump_dir is not None:
            c = np.load(os.path.join(d, "C_numba.npy" if out["kind"] == "reference" else "C_port.npy"))
            rows = dump_rows(c.shape[0], c.shape[1])
            write_outputs(dump_dir, c[rows], rows)
        return out
    finally:
        shutil.rmtree(d, ignore_errors=True)


# ---- gather of the row-sharded B: one interface, two transports ---------------------------------------------------------
class NcclGather:
    """dist.all_gather_into_tensor on a side stream into a double buffer (SM-based NCCL kernels)."""

    def __init__(self, torch, dist, shard, n_buffers=2):
        self.torch, self.dist, self.shard = torch, dist, shard
        world = dist.get_world_size()
        self.comm = torch.cuda.Stream(device=shard.device)
        self.buffers = [torch.empty((shard.shape[0] * world, shard.shape[1]), dtype=shard.dtype, device=shard.device)
                        for _ in range(n_buffers)]
        self._done = [torch.cuda.Event() for _ in range(n_buffers)]
        self._released = [torch.cuda.Event() for _ in range(n_buffers)]
        for e in self._released:
            e.record()

    def gather(self, slot):
        with self.torch.cuda.stream(self.comm):
            self.comm.wait_event(self._released[slot])
            self.dist.all_gather_into_tensor(self.buffers[slot], self.shard)
            self._done[slot].record(self.comm)

    def acquire(self, slot):
        self.torch.cuda.current_stream().wait_event(self._done[slot])
        return self.buffers[slot]

    def release(self, slot):
        self._released[slot].record(self.torch.cuda.current_stream())

    def close(self):
        pass


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    M = K = args.rows
    ncols = args.ncols

    if args.impl == "reference":
        return reference_arm(args, rank, local_rank, world)

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the sparse_b200 hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    from sparse_b200 import _dist as SD

    # host threads (the library's staging pool, pinned first-touch) live on the GPU's NUMA node, split between ranks
    numa = SD.bind_to_gpu_numa(local_rank, local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", world))) \
        if not args.no_numa else None
    from sparse_b200 import _kernels as Kn
    from sparse_b200 import _lib

    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    _lib.load()
    if args.variant or args.unroll:
        Kn.spmm_set_variant(args.variant or 1, args.unroll or 8)

    def allmax(x):
        if world == 1:
            return float(x)
        t = torch.tensor([float(x)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allmin(x):
        return -allmax(-float(x))

    def allsum(x):
        if world == 1:
            return float(x)
        t = torch.tensor([float(x)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    vals, cols, indptr, _g = gen_A(torch, M, K, args.nnz, A_SEED + rank, dev)
    B = gen_B(torch, K, ncols, B_SEED, dev)
    nnz = int(vals.numel())
    C = torch.empty((M, ncols), dtype=torch.float32, device=dev)

    # N > 1: every step needs its own gather of the row-sharded B.  The gather of step i+1 runs on side streams into
    # the other half of a double buffer while K1 of step i runs (events order buffer reuse: gather(i+2) waits for
    # K1(i), K1(i) waits for gather(i)).
    gatherer, gather_kind = None, None
    if world > 1:
        assert K % world == 0
        shard_rows = K // world
        if args.gather == "ce":
            try:
                gatherer = SD.PeerGather(shard_rows, ncols, np.float32)
                gatherer.shard.copy_(B[rank * shard_rows:(rank + 1) * shard_rows])
                gatherer.publish()
                gather_kind = "copy engines (CUDA IPC peer buffers, cudaMemcpyAsync pull over NVLink; csrc/peer.cu)"
            except Exception as e:  # loud, and visible in the JSON line
                print(f"[bench rank {rank}] PeerGather unavailable ({e}); using the NCCL all-gather", file=sys.stderr)
                gatherer = None
        ok = allmin(1.0 if gatherer is not None or args.gather != "ce" else 0.0)
        if args.gather == "ce" and ok < 1.0 and gatherer is not None:
            gatherer.close()
            gatherer = None
        if gatherer is None:
            gatherer = NcclGather(torch, dist, B[rank * shard_rows:(rank + 1) * shard_rows].clone())
            gather_kind = "NCCL all_gather_into_tensor on a side stream (SM kernels)"

    def make_steps(a, Cout, Msub, g, B_direct):
        """n pipelined steps of (gather ->) K1 on the row block `a` = (vals, cols, indptr)."""
        av, ac, ap = a

        def run(n, kev=None):
            if g is not None:
                g.gather(0)
            for i in range(n):
                slot = i % 2
                if g is not None:
                    if i + 1 < n:
                        g.gather((i + 1) % 2)
                    Bf = g.acquire(slot)
                else:
                    Bf = B_direct
                if kev is not None:
                    kev[i][0].record()
                Kn.spmm_csr_dense(av, ac, ap, Bf, Msub, K, ncols, out=Cout)
                if kev is not None:
                    kev[i][1].record()
                if g is not None:
                    g.release(slot)
        return run

    def timed(run, steps, clock_index=None):
        """K steps between barrier + synchronize on both sides, CUDA events on the launching stream, max over ranks."""
        kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        clk = clock_index  # a ClockSampler that is already running (started before the warm-up), or None
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.time()
        t0.record()
        run(steps, kev)
        t1.record()
        torch.cuda.synchronize()
        if clk:
            clk.window = (w0, time.time())
            clk.__exit__()
        total = allmax(t0.elapsed_time(t1))
        kern = sum(a.elapsed_time(b) for a, b in kev) / steps
        if world > 1:
            dist.barrier()
        return total / steps, kern, clk

    run_steps = make_steps((vals, cols, indptr), C, M, gatherer, B)
    # clocks / throttle reasons DURING the timed region: one nvidia-smi in loop mode on rank 0 only (eight of them slow
    # each other down), started before the warm-up so that it is up when the region starts; samples are time-stamped
    # and only those inside the region are summarised
    sampler = None
    if rank == 0:
        sampler = ClockSampler(local_rank)
        sampler.__enter__()
    run_steps(max(args.warmup, 3))
    torch.cuda.synchronize()

    # the distributed product is checked, not assumed: C from the gathered operand == C from the local copy of B
    dist_check = None
    if world > 1:
        gatherer.gather(0)
        Bf = gatherer.acquire(0)
        C_g = Kn.spmm_csr_dense(vals, cols, indptr, Bf, M, K, ncols)
        gatherer.release(0)
        C_l = Kn.spmm_csr_dense(vals, cols, indptr, B, M, K, ncols)
        same = bool(torch.equal(Bf, B)) and bool(torch.equal(C_g.view(torch.int32), C_l.view(torch.int32)))
        dist_check = bool(allmin(1.0 if same else 0.0) == 1.0)
        del C_g, C_l
        torch.cuda.synchronize()

    launches0 = _lib.launch_count()
    ms_per_step, kern_ms, clk = timed(run_steps, args.steps, clock_index=sampler)
    launches = _lib.launch_count() - launches0
    if args.dump_outputs is not None:  # C still holds the last timed step; the blocks below reuse it
        rows = dump_rows(M, ncols, share=world)
        write_outputs(args.dump_outputs, C[torch.from_numpy(rows).to(dev)].cpu().numpy(), rows,
                      suffix=f"_rank{rank}" if world > 1 else "")
    nnz_all = allsum(nnz)
    value = nnz_all / (ms_per_step * 1e-3) / 1e9

    peak, peak_src = peaks()
    alg = algorithmic_bytes(nnz, M, ncols)
    achieved = alg / (kern_ms * 1e-3) / 1e9
    roof = {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
            "frac": round(achieved / peak, 4), "traffic": known_traffic(ncols),
            "kernel": {0: "spmm_csr_dense_dyn_kernel<f32,i32,VEC4,G32,U8>", 1: "spmm_csr_dense_dyn_kernel<f32,i32,VEC4,G32,U8>",
                       2: "spmm_csr_dense_tma_kernel<f32,i32>", 3: "spmm_csr_dense_kernel<f32,i32,VEC4,G32,U8>"}.get(
                           args.variant, "spmm_csr_dense_dyn_kernel<f32,i32,VEC4,G32,U8>"),
            "kernel_ms": round(kern_ms, 4), "algorithmic_bytes_per_launch": alg,
            "bytes_per_nnz_model": round(alg / nnz, 2), "peak_source": peak_src,
            "compulsory_bytes_per_launch": nnz * 8 + (M + 1) * 4 + K * ncols * 4 + M * ncols * 4,
            "traffic_source": "profiles/k1_traffic.json (one ncu --set full capture of this kernel at this size; "
                              "a constant, not re-measured per run)"}

    # ---- strong scaling of the NAMED problem (1e8 nnz in total) over the N GPUs ----------------------------------------
    strong = None
    if world > 1 and not args.no_strong:
        if rank == 0:
            sv, sc, sp_ = vals, cols, indptr
        else:
            sv, sc, sp_, _ = gen_A(torch, M, K, args.nnz, A_SEED, dev)
        ip64 = sp_.to(torch.int64)
        tot = int(ip64[-1].item())
        targets = torch.tensor([tot * r // world for r in range(1, world)], device=dev, dtype=torch.int64)
        cuts = [0] + [int(x) for x in torch.searchsorted(ip64, targets).tolist()] + [M]
        r0, r1 = cuts[rank], cuts[rank + 1]
        lo, hi = int(ip64[r0].item()), int(ip64[r1].item())
        blk = (sv[lo:hi], sc[lo:hi], (ip64[r0:r1 + 1] - lo).to(torch.int32).contiguous())
        Cb = C[: r1 - r0]
        res = {}
        for name, g in (("replicated_B", None), ("sharded_B", gatherer)):
            run = make_steps(blk, Cb, r1 - r0, g, B)
            run(max(args.warmup, 3))
            ms, kms, _ = timed(run, args.steps)
            res[name] = {"ms_per_step": round(ms, 4), "GNNZ/s": round(tot / ms / 1e6, 4),
                         "kernel_ms_rank0": round(kms, 4)}
        # the row block equals the same rows of the single-GPU product of the whole matrix
        full = Kn.spmm_csr_dense(sv, sc, sp_, B, M, K, ncols)
        same = bool(torch.equal(full[r0:r1].view(torch.int32), Cb.view(torch.int32)))
        del full
        res["row_blocks_bit_exact_vs_single_gpu_product"] = bool(allmin(1.0 if same else 0.0) == 1.0)
        res["problem"] = f"C2 fixed: {M}x{K}, nnz={tot} in total, nnz-balanced row blocks (cut on indptr)"
        res["collective"] = {"replicated_B": "none", "sharded_B": gather_kind}
        res["block_nnz_min_max"] = [int(allmin(hi - lo)), int(allmax(hi - lo))]
        strong = res
        del blk, Cb
        if rank != 0:
            del sv, sc, sp_
        torch.cuda.synchronize()

    # ---- e2e through the host-buffer C-ABI call (rank-local; N>1 reports the aggregate) ------------
    e2e = None
    narrowing = SD.configure_host_staging(int(os.environ.get("LOCAL_WORLD_SIZE", world)))
    if not args.no_e2e:
        h_vals = vals.cpu().pin_memory()
        h_cols = cols.cpu().to(torch.int64).pin_memory()
        h_ptr = indptr.cpu().to(torch.int64).pin_memory()
        h_B = B.cpu().pin_memory()
        h_C = torch.empty((M, ncols), dtype=torch.float32).pin_memory()
        import sparse_b200 as sp

        npv = (h_vals.numpy(), h_cols.numpy(), h_ptr.numpy(), h_B.numpy())
        esteps = args.steps

        def e2e_step():
            # the call a user of the reference makes: host arrays in, np.ndarray out (H2D + K1 + D2H inside)
            A = sp.GCXS((npv[0], npv[1], npv[2]), shape=(M, K), compressed_axes=(0,))
            return sp.tensordot(A, npv[3], axes=1)

        for _ in range(3):  # warm-up (pinned result pool, scratch pool, page mapping)
            h_res = e2e_step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(esteps):
            h_res = e2e_step()
        torch.cuda.synchronize()
        e_ms = allmax((time.perf_counter() - t0) * 1e3 / esteps)
        h_C.copy_(torch.from_numpy(h_res))
        # bytes that cross PCIe per step: values, column indices (int64 on the host, narrowed to int32 by the
        # library's host thread pool into pinned staging before the copy), int64 indptr, B; and C coming back
        host_in = int(h_vals.numel() * 4 + h_cols.numel() * 8 + h_ptr.numel() * 8 + h_B.numel() * 4)
        h2d = int(h_vals.numel() * 4 + h_cols.numel() * 4 + h_ptr.numel() * 8 + h_B.numel() * 4)
        d2h = int(h_C.numel() * 4)
        e2e = {"value": round(nnz_all / (e_ms * 1e-3) / 1e9, 4), "unit": "GNNZ/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "host_input_bytes_per_step": host_in, "ms_per_step": round(e_ms, 3),
               "steps": esteps,
               "api": "sparse_b200.tensordot(GCXS(host arrays, int64 indices), np.ndarray) -> np.ndarray "
                      "(b2s_spmm_csr_dense_host: int64->int32 index narrowing on the " + narrowing + " + 3-stream "
                      "H2D/K1/D2H pipeline, pinned buffers)", "index_narrowing": narrowing}
        if narrowing == "device":  # the raw int64 indices cross the bus
            e2e["h2d_bytes_per_step"] = host_in
        if world > 1:  # the other staging mode, for the record
            _lib.load().b2s_spmm_host_set_threads(_lib.i32(-1 if narrowing == "device" else 0))
            for _ in range(2):
                e2e_step()
            torch.cuda.synchronize()
            dist.barrier()
            t0 = time.perf_counter()
            for _ in range(esteps):
                e2e_step()
            torch.cuda.synchronize()
            alt_ms = allmax((time.perf_counter() - t0) * 1e3 / esteps)
            e2e["other_staging_mode"] = {"index_narrowing": "host" if narrowing == "device" else "device",
                                         "ms_per_step": round(alt_ms, 3)}
            SD.configure_host_staging(int(os.environ.get("LOCAL_WORLD_SIZE", world)))
        C_ref = Kn.spmm_csr_dense(vals, cols, indptr, B, M, K, ncols, out=C)
        e2e["matches_device_path"] = bool(allmin(1.0 if torch.equal(h_C.to(dev), C_ref) else 0.0) == 1.0)
        del h_vals, h_cols, h_ptr, h_B, h_C, npv, h_res

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        rows_sample = min(M, args.cpu_rows or CPU_ROWS)
        Kn.spmm_csr_dense(vals, cols, indptr, B, M, K, ncols, out=C)
        torch.cuda.synchronize()
        cpu = cpu_legs(vals, cols, indptr, B, K, ncols, rows_sample, steps=3, warmup=1,
                       gpu_rows=C[:rows_sample].cpu().numpy())

    configs = None
    if rank == 0 and world == 1 and not args.no_configs:
        del vals, cols, indptr, B, C
        torch.cuda.empty_cache()
        try:
            from tools import bench_configs

            configs = bench_configs.run(compact=True)
        except Exception as e:  # never lose the headline line to a side block
            configs = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        cfg = workload_config(M, K, nnz, ncols, world, gather_kind)
        if numa:
            cfg["host_affinity"] = numa
        if dist_check is not None:
            cfg["distributed_product_bit_exact_vs_local_B"] = dist_check
        line = {
            "metric": "CSR x dense tensordot throughput (GNNZ/s)", "value": round(value, 4), "unit": "GNNZ/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms_per_step, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg, "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches),
            "clocks": clk.summary(),
        }
        if strong is not None:
            line["strong"] = strong
        if configs is not None:
            line["configs"] = configs
        print(json.dumps(line), flush=True)
    if world > 1:
        if gatherer is not None:
            gatherer.close()
        dist.destroy_process_group()


def workload_config(M, K, nnz, ncols, world, gather_kind=None):
    """The `config` object of the JSON line -- identical for the product arm and the reference arm."""
    return {"workload": f"C2: GCXS/CSR({M}x{K}, nnz={nnz} per GPU, uniform) @ dense({K}x{ncols}) fp32 -> dense",
            "index_dtype_device": "int32", "l2": "inputs>L2 (2.2 GB operands vs 126 MB L2), no flush",
            "parallelism": ("1-D row blocks of A per GPU; B row-sharded, gathered EVERY step into a double buffer on "
                            "side streams (overlaps the previous step's K1): " + str(gather_kind))
            if world > 1 else "single GPU",
            "exact_order": True}


def reference_arm(args, rank, local_rank, world):
    """--impl reference: the reference's OWN implementation of the path on the host cores.

    oracle/_ref holds the unmodified pydata/sparse (oracle/make_ref.sh); a worker process imports it and times
    `sparse.tensordot(GCXS, ndarray, axes=1)` -> _dot_csr_ndarray (_common.py:95, 720-755), a single-threaded numba
    kernel (cores = 1 by construction), on a bounded sample of the GPU arm's own arrays: the first CPU_ROWS rows of
    rank 0's A (same seeded generator, run on cuda:0 when the box has one -- input generation only) times the full B.
    The sample and the thread counts do not depend on the launcher.  A second, labelled figure comes from the OpenMP
    port (fixed 32 threads).  Only rank 0 works; the other ranks exit 0."""
    if rank != 0:
        return
    import torch

    M = K = args.rows
    ncols = args.ncols
    rows_sample = min(M, args.cpu_rows or CPU_ROWS)
    dev = torch.device("cuda", local_rank) if torch.cuda.is_available() else torch.device("cpu")
    if dev.type == "cuda":
        vals, cols, indptr, _ = gen_A(torch, M, K, args.nnz, A_SEED, dev)
    else:  # authoring container: same distribution, host generator, only the sampled rows
        vals, cols, indptr, _ = gen_A(torch, rows_sample, K, args.nnz // max(1, M // rows_sample), A_SEED, dev)
    B = gen_B(torch, K, ncols, B_SEED, dev)
    cpu = cpu_legs(vals, cols, indptr, B, K, ncols, rows_sample, steps=args.steps, warmup=max(args.warmup, 1),
                   dump_dir=args.dump_outputs)
    val = cpu["value"]
    n = int(indptr[rows_sample].item())
    line = {
        "impl": "reference", "metric": "CSR x dense tensordot throughput (GNNZ/s)", "value": val,
        "unit": "GNNZ/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 1),
        "ms_per_step": round(n / val / 1e6, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(M, K, args.nnz, ncols, world, "n/a (CPU reference)"),
        "cpu_baseline": cpu,
        "e2e": {"value": val, "unit": "GNNZ/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "inputs_generated_on": str(dev),
    }
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
