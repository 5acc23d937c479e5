"""Multi-GPU execution of the hot path: one process per GPU, 1-D row blocks of the left operand.

The path shards naturally along the first (row) axis of the left operand: output rows are independent, so the
only exchange is making the right operand visible to every rank (SURVEY.md s8(e)):

* ``tensordot_rowblock``   C_r = A_r @ B:  A_r is this rank's nnz-balanced row block, B arrives row-sharded and is
  all-gathered over NCCL/NVLink (``dist.all_gather_into_tensor``) before the local K1 kernel.
* ``spgemm_rowblock``      C_r = A_r @ B for sparse B: B's CSR arrays are all-gathered (variable sizes, padded).
* ``sddmm_rowblock``       mask row block x local rows of `a`; `b` (K x N) arrives column-sharded and is gathered.
* ``masked_matmul_rowblock`` sparse mask row block x local rows of sparse `a`; `b`'s row blocks (CSR) are gathered.

No reduction collective is needed for row blocking (a reduce-scatter would only appear if the CONTRACTION axis
were split, which doubles the dense traffic; see DESIGN.md).  Host logic is backend-agnostic: the `gloo` tests
run it with world_size 2 on CPU tensors.
"""
from __future__ import annotations

import numpy as np

from . import _device as D
from . import _kernels as Kn


def nnz_balanced_splits(indptr, world: int):
    """Row boundaries r_0=0 <= r_1 <= ... <= r_world=M such that every block holds ~nnz/world stored entries
    (split points are chosen on indptr, not on the row count)."""
    ip = np.asarray(indptr, dtype=np.int64)
    M = len(ip) - 1
    nnz = int(ip[-1]) if M >= 0 and len(ip) else 0
    bounds = [0]
    for r in range(1, world):
        target = nnz * r // world
        cut = int(np.searchsorted(ip, target, side="left"))
        cut = min(max(cut, bounds[-1]), M)
        bounds.append(cut)
    bounds.append(M)
    return bounds


def row_block(data, indices, indptr, r0: int, r1: int):
    """Rows [r0, r1) of a CSR triple (host arrays); indptr rebased to 0."""
    ip = np.asarray(indptr)
    lo, hi = int(ip[r0]), int(ip[r1])
    return data[lo:hi], indices[lo:hi], (ip[r0:r1 + 1] - ip[r0])


def _dist():
    import torch.distributed as dist

    return dist


def all_gather_rows(shard, group=None):
    """Concatenate equally sized row shards of a dense operand along axis 0 (one all-gather)."""
    dist = _dist()
    t = D.torch()
    world = dist.get_world_size(group)
    if world == 1:
        return shard
    shard = shard.contiguous()
    out = t.empty((shard.shape[0] * world,) + tuple(shard.shape[1:]), dtype=shard.dtype, device=shard.device)
    dist.all_gather_into_tensor(out, shard, group=group)
    return out


def all_gather_sizes(values, group=None):
    """All-gather a short list of host integers (one collective, one host sync): returns a (world, len) int64 array."""
    dist = _dist()
    t = D.torch()
    world = dist.get_world_size(group)
    dev = D.device()
    mine = t.tensor([int(v) for v in values], dtype=t.int64, device=dev)
    out = t.empty((world, len(values)), dtype=t.int64, device=dev)
    dist.all_gather_into_tensor(out, mine.reshape(1, -1), group=group)
    return out.cpu().numpy()


def all_gather_padded(x, sizes, group=None):
    """All-gather 1-D tensors whose lengths `sizes` (host, one per rank) are already known: ONE collective into a
    (world, max) buffer; returns the per-rank views (no copy).  No size exchange, no host sync."""
    dist = _dist()
    t = D.torch()
    world = dist.get_world_size(group)
    mx = max(int(v) for v in sizes) if len(sizes) else 0
    mx = max(mx, 1)
    if int(x.shape[0]) == mx:
        pad = x.contiguous()
    else:
        pad = t.zeros(mx, dtype=x.dtype, device=x.device)
        pad[: x.shape[0]] = x
    out = t.empty((world, mx), dtype=x.dtype, device=x.device)
    dist.all_gather_into_tensor(out, pad.reshape(1, mx), group=group)
    return [out[r, : int(sizes[r])] for r in range(world)]


def all_gather_varlen(x, group=None):
    """All-gather 1-D tensors of different lengths: returns (list of per-rank tensors)."""
    dist = _dist()
    world = dist.get_world_size(group)
    if world == 1:
        return [x]
    sizes = all_gather_sizes([int(x.shape[0])], group)[:, 0]
    return all_gather_padded(x, sizes, group)


class _RawDeviceBuffer:
    """`__cuda_array_interface__` holder for a cudaMalloc'ed / IPC-mapped pointer (torch.as_tensor wraps it, no copy)."""

    def __init__(self, ptr: int, shape, np_dtype):
        self.__cuda_array_interface__ = {"shape": tuple(int(x) for x in shape), "typestr": np.dtype(np_dtype).str,
                                         "data": (int(ptr), False), "version": 2, "strides": None}


class PeerGather:
    """All-gather of equal row shards of a dense operand by COPY ENGINES over NVLink (csrc/peer.cu).

    Every rank owns an IPC-exported shard buffer (`.shard`, a torch view the caller fills) and `n_buffers` full-size
    receive buffers; `gather(slot)` pulls all world shards into buffer `slot` with cudaMemcpyAsync on side streams --
    DMA, no kernel -- so the exchange takes no SM and no issue slot from the DRAM-bound product kernel it overlaps
    (an SM-based NCCL all-gather slows K1 by 5.6 % at N = 8, profiles/r01).  Ordering inside a rank is by events
    (`gather` waits for `release(slot)`, consumers call `acquire(slot)`); ordering ACROSS ranks (a peer's shard must be
    complete before it is pulled) is the caller's: `publish()` = local synchronise + barrier after writing `.shard`.
    """

    def __init__(self, shard_rows: int, ncols: int, dtype, group=None, n_buffers: int = 2, n_streams: int = 2):
        import ctypes

        from . import _lib

        dist = _dist()
        t = D.torch()
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.dtype = np.dtype(dtype)
        self.shard_rows, self.ncols = int(shard_rows), int(ncols)
        self.shard_bytes = self.shard_rows * self.ncols * self.dtype.itemsize
        self._lib = lib = _lib.load()
        dev = t.device("cuda", t.cuda.current_device())
        p = ctypes.c_void_p()
        _lib.check(lib.b2s_peer_alloc(ctypes.byref(p), _lib.i64(self.shard_bytes)), "b2s_peer_alloc")
        self._own = int(p.value)
        h = (ctypes.c_ubyte * 64)()
        _lib.check(lib.b2s_peer_export(_lib.vp(self._own), h), "b2s_peer_export")
        handles = [None] * self.world
        dist.all_gather_object(handles, bytes(h), group=group)
        self._ptrs, self._opened = [], []
        for r, hb in enumerate(handles):
            if r == self.rank:
                self._ptrs.append(self._own)
                continue
            q = ctypes.c_void_p()
            buf = (ctypes.c_ubyte * 64).from_buffer_copy(hb)
            _lib.check(lib.b2s_peer_open(buf, ctypes.byref(q)), f"b2s_peer_open(rank {r})")
            self._ptrs.append(int(q.value))
            self._opened.append(int(q.value))
        self._ptr_arr = (ctypes.c_void_p * self.world)(*self._ptrs)
        self.shard = t.as_tensor(_RawDeviceBuffer(self._own, (self.shard_rows, self.ncols), self.dtype), device=dev)
        self.buffers = [t.empty((self.shard_rows * self.world, self.ncols), dtype=self.shard.dtype, device=dev)
                        for _ in range(n_buffers)]
        self.streams = [t.cuda.Stream(device=dev) for _ in range(n_streams)]
        self._stream_arr = (ctypes.c_void_p * n_streams)(*[s.cuda_stream for s in self.streams])
        self._done = [[t.cuda.Event() for _ in self.streams] for _ in range(n_buffers)]
        self._released = [t.cuda.Event() for _ in range(n_buffers)]
        for e in self._released:
            e.record()

    def publish(self):
        """The local shard is final: make it visible to the peers (device sync + barrier)."""
        D.torch().cuda.synchronize()
        _dist().barrier(group=self.group)

    def gather(self, slot: int):
        """Start pulling every rank's shard into buffers[slot] (returns immediately; copy engines do the work)."""
        from . import _lib

        for s in self.streams:
            s.wait_event(self._released[slot])
        _lib.check(self._lib.b2s_peer_gather(_lib.vp(D.ptr(self.buffers[slot])), self._ptr_arr, _lib.i32(self.world),
                                             _lib.i32(self.rank), _lib.i64(self.shard_bytes), self._stream_arr,
                                             _lib.i32(len(self.streams))), "b2s_peer_gather")
        for s, e in zip(self.streams, self._done[slot]):
            e.record(s)

    def acquire(self, slot: int, stream=None):
        """Make `stream` (default: current) wait until buffers[slot] holds the gathered operand; returns it."""
        stream = stream or D.torch().cuda.current_stream()
        for e in self._done[slot]:
            stream.wait_event(e)
        return self.buffers[slot]

    def release(self, slot: int, stream=None):
        """The consumer launched on `stream` is the last reader of buffers[slot]; the next gather(slot) waits for it."""
        self._released[slot].record(stream or D.torch().cuda.current_stream())

    def close(self):
        D.torch().cuda.synchronize()
        _dist().barrier(group=self.group)  # nobody is still pulling from the buffer freed below
        for q in self._opened:
            self._lib.b2s_peer_close(ctypes_vp(q))
        self._opened = []
        if self._own:
            self.shard = None
            self._lib.b2s_peer_free(ctypes_vp(self._own))
            self._own = 0


def ctypes_vp(x):
    import ctypes

    return ctypes.c_void_p(int(x))


_numa_note = [""]


def gpu_numa_cpus(device_index: int):
    """CPUs of the NUMA node the GPU hangs off (sysfs; None when it cannot be determined)."""
    import os

    bus = None
    try:
        import subprocess

        # nvidia-smi prints "00000000:1B:00.0" (8-digit PCI domain); CUDA_VISIBLE_DEVICES renumbers devices, so ask
        # the runtime for the UUID-independent PCI id of the ordinal CUDA uses
        t = D.torch()
        props = t.cuda.get_device_properties(device_index)
        dom = getattr(props, "pci_domain_id", None)
        b_ = getattr(props, "pci_bus_id", None)
        d_ = getattr(props, "pci_device_id", None)
        if isinstance(b_, int) and isinstance(d_, int):
            bus = f"{int(dom or 0):04x}:{b_:02x}:{d_:02x}.0"
        elif isinstance(b_, str):
            bus = b_
        if bus is None:
            bus = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i",
                                  str(device_index)], capture_output=True, text=True, timeout=10).stdout.strip()
    except Exception:
        bus = None
    try:
        if not bus:
            return None
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:  # nvidia-smi prints an 8-digit PCI domain, sysfs uses 4
            bus = bus[4:]
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            _numa_note[0] = f"sysfs numa_node of {bus} is {node} (no NUMA topology visible in this container / VM)"
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            spec = f.read().strip()
        cpus = []
        for part in spec.split(","):
            lo, _, hi = part.partition("-")
            cpus.extend(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in allowed]
        return (node, cpus) if cpus else None
    except Exception as e:
        _numa_note[0] = f"{type(e).__name__}: {e}"
        return None


def configure_host_staging(local_world: int):
    """Host-buffer products (`tensordot(GCXS(host arrays), ndarray)`) narrow int64 indices to int32 on the host before
    the H2D copy: fewer PCIe bytes (1.32 instead of 1.72 GB at C2) for one extra pass over host memory.  One rank per
    GPU with 4+ ranks on a box makes HOST DRAM the bottleneck (every rank streams ~2.5 GB per product through it), so the
    extra pass is switched off there and the raw int64 indices are uploaded and narrowed on the device.  Returns the
    setting ("host" | "device")."""
    from . import _lib

    lib = _lib.load()
    if local_world >= 4:
        lib.b2s_spmm_host_set_threads(_lib.i32(0))
        return "device"
    lib.b2s_spmm_host_set_threads(_lib.i32(-1))
    return "host"


def bind_to_gpu_numa(device_index: int, local_rank: int = 0, local_world: int = 1):
    """Pin this process (and every thread it starts afterwards: the library's host thread pool, pinned-staging
    first-touch) to its GPU's NUMA node, split evenly between the ranks whose GPUs share that node.  Host staging of
    the host-buffer product is memory-bound; with 8 ranks and no affinity the ranks of GPUs 4-7 stage through the
    other socket.  Returns a description (dict) or None when the topology is not visible."""
    import os

    got = gpu_numa_cpus(device_index)
    if got is None:
        return {"numa_node": None, "note": _numa_note[0] or "GPU PCI id not found"}
    node, cpus = got
    # ranks that share the node: assume local ranks map to device indices 0..local_world-1
    sharers = [r for r in range(local_world) if (gpu_numa_cpus(r) or (None,))[0] == node] or [local_rank]
    k = sharers.index(local_rank) if local_rank in sharers else 0
    per = max(1, len(cpus) // len(sharers))
    mine = cpus[k * per:(k + 1) * per] or cpus
    try:
        os.sched_setaffinity(0, mine)
    except Exception:
        return None
    return {"numa_node": node, "cpus": len(mine), "first_cpu": mine[0], "ranks_on_node": len(sharers)}


def tensordot_rowblock(a_local, b_shard, group=None, out=None):
    """Local block of ``A @ B`` (dense result rows owned by this rank).

    a_local : 2-D GCXS (compressed_axes=(0,)) holding this rank's row block of A (all K columns).
    b_shard : dense device tensor, this rank's K/world rows of B (equal shards).
    """
    from ._dot import _csr_arrays, _dot_dtype

    B = all_gather_rows(b_shard, group)
    M, K = a_local.shape
    assert B.shape[0] == K, (B.shape, K)
    dtr = _dot_dtype(a_local.dtype, D.np_dtype(B))
    ad, ai, ap = _csr_arrays(a_local, dtr)
    return Kn.spmm_csr_dense(ad, ai, ap, Kn.cast(B, dtr), M, K, int(B.shape[1]), out=out)


def gather_csr_rows(b_local, group=None):
    """All-gather a row-sharded CSR operand (each rank owns a block of consecutive rows): one exchange of the block
    sizes (the only host sync), then one padded collective per array; the row pointers are rebased with the prefix sums
    of the exchanged nnz counts (host integers -- no device read-backs)."""
    from ._gcxs import GCXS

    t = D.torch()
    dist = _dist()
    world = dist.get_world_size(group)
    data, indices, indptr = b_local._dev()
    if world == 1:
        return b_local
    sizes = all_gather_sizes([int(data.shape[0]), int(indptr.shape[0])], group)
    nnzs, ptr_lens = sizes[:, 0], sizes[:, 1]
    datas = all_gather_padded(data, nnzs, group)
    idxs = all_gather_padded(indices.to(t.int64), nnzs, group)
    ptrs = all_gather_padded(indptr.to(t.int64), ptr_lens, group)
    out_ptr, base = [], 0
    for r in range(world):
        p = ptrs[r]
        out_ptr.append((p if r == 0 else p[1:]) + base)
        base += int(nnzs[r])
    full_ptr = t.cat(out_ptr)
    rows = int(full_ptr.shape[0]) - 1
    return GCXS((t.cat(datas), t.cat(idxs), full_ptr), shape=(rows, b_local.shape[1]), compressed_axes=(0,))


def spgemm_rowblock(a_local, b_local, group=None):
    """Local row block of ``A @ B`` for sparse operands: B's row blocks are all-gathered, then K4 runs locally."""
    from ._dot import _dot

    B = gather_csr_rows(b_local, group)
    assert a_local.shape[1] == B.shape[0]
    return _dot(a_local, B)


def all_to_all_varlen(chunks, group=None):
    """Send chunks[q] (1-D, same dtype) to rank q; returns the list of chunks received (one per source rank).  One
    exchange of the chunk lengths (host sync), then `all_to_all_single` with uneven splits (NCCL); backends without it
    (gloo on CPU, used by the tests) gather every chunk and keep their own."""
    dist = _dist()
    t = D.torch()
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    if world == 1:
        return [chunks[0]]
    send_sizes = [int(c.shape[0]) for c in chunks]
    table = all_gather_sizes(send_sizes, group)  # table[src, dst]
    recv_sizes = [int(table[src, rank]) for src in range(world)]
    send = t.cat(chunks) if sum(send_sizes) else chunks[0][:0]
    recv = t.empty(sum(recv_sizes), dtype=send.dtype, device=send.device)
    try:
        if dist.get_backend(group) != "nccl":
            raise RuntimeError("no all_to_all_single")
        dist.all_to_all_single(recv, send, output_split_sizes=recv_sizes, input_split_sizes=send_sizes, group=group)
    except RuntimeError:
        everything = all_gather_padded(send, [int(table[r].sum()) for r in range(world)], group)
        pieces = []
        for src in range(world):
            lo = int(table[src, :rank].sum())
            pieces.append(everything[src][lo:lo + recv_sizes[src]])
        recv = t.cat(pieces) if pieces else recv
    out, at = [], 0
    for n in recv_sizes:
        out.append(recv[at:at + n])
        at += n
    return out


def spgemm_ksplit(a_colblock, b_rowblock, group=None):
    """``A @ B`` with the CONTRACTION axis split (the alternative to row blocking, SURVEY.md s8(e)): rank r holds the
    column block A[:, K_r] (all M rows) and the matching row block B[K_r, :]; every rank multiplies its pair into a
    sparse partial over ALL rows, the partials' row blocks are exchanged (all-to-all of (key, value) fragments -- the
    "reduce-scatter of output rows": NCCL has no sparse reduce-scatter) and each rank sums the `world` fragments of its
    row block (device sort + duplicate summation).  Returns this rank's block of consecutive output rows as a canonical
    COO (columns ascending; partial sums are added across K blocks, so values equal the row-blocked product to
    rounding, not bit for bit -- which is one reason row blocking is the production form; the other is traffic: the
    partials hold up to `world` x the output entries)."""
    from ._coo import COO
    from ._dot import _dot

    dist = _dist()
    t = D.torch()
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    M, N = int(a_colblock.shape[0]), int(b_rowblock.shape[1])
    part = _dot(a_colblock, b_rowblock)  # GCXS (compressed rows), M x N
    data, indices, indptr = part._dev()
    nnz = int(data.shape[0])
    rows = Kn.rows_from_indptr(indptr, nnz, np.int64)
    keys = Kn.linearize(t.stack([rows, indices.to(t.int64)]), [N, 1])
    bounds = [M * q // world for q in range(world + 1)]
    cut = D.download(indptr[t.as_tensor(bounds, device=indptr.device)]).astype(np.int64)  # entries before each block
    k_in = all_to_all_varlen([keys[int(cut[q]):int(cut[q + 1])] for q in range(world)], group)
    v_in = all_to_all_varlen([data[int(cut[q]):int(cut[q + 1])] for q in range(world)], group)
    r0, r1 = bounds[rank], bounds[rank + 1]
    allk = t.cat(k_in) - r0 * N
    allv = t.cat(v_in)
    shape = (r1 - r0, N)
    if int(allk.shape[0]) == 0:
        return COO(np.zeros((2, 0), dtype=np.intp), np.empty(0, dtype=part.dtype), shape=shape)
    return COO(Kn.unravel(allk, shape, np.int64), allv, shape=shape, has_duplicates=True, sorted=False, prune=True)


def sddmm_rowblock(s_local, a_local, b_cols_shard, group=None):
    """Local row block of ``s * (a @ b)``: `b` arrives column-sharded (K x N/world) and is gathered as b^T rows."""
    from ._fused import sddmm

    bt_shard = Kn.transpose_dense(b_cols_shard)  # (N/world, K)
    Bt = all_gather_rows(bt_shard, group)        # (N, K)
    return sddmm(s_local, a_local, Bt, b_transposed=True)


def masked_matmul_rowblock(s_local, a_local, b_local, group=None):
    """Local row block of ``s * (a @ b)`` for sparse operands: `s` and `a` hold the same block of rows, `b` is
    row-sharded as CSR blocks that are all-gathered, then K10 runs locally."""
    from ._fused import masked_matmul

    B = gather_csr_rows(b_local, group)
    return masked_matmul(s_local, a_local, B)


# ---- element-wise operations and reductions: range partition on the leading coordinate (SURVEY.md s8(e)) -------------
def leading_splits(arrays, world: int):
    """Boundaries on the LEADING axis shared by every operand such that each rank holds ~1/world of the stored
    entries of all operands together (operands whose leading extent is 1 are broadcast there and are not split)."""
    ext = max(a.shape[0] for a in arrays)
    counts = np.zeros(ext, dtype=np.int64)
    for a in arrays:
        if a.shape[0] != ext:
            continue
        lead = a.coords[0] if a.nnz else np.empty(0, dtype=np.int64)
        counts += np.bincount(lead, minlength=ext)
    return nnz_balanced_splits(np.concatenate([[0], np.cumsum(counts)]), world)


def leading_block(x, r0: int, r1: int):
    """Entries of COO `x` whose leading coordinate lies in [r0, r1) (one pass of the slice kernel); an operand that is
    broadcast on the leading axis (extent 1) is replicated."""
    if x.shape[0] == 1 and r1 - r0 != 1:
        return x
    return x[r0:r1]


def elemwise_leading(func, *local_blocks, **kwargs):
    """Local block of ``elemwise(func, *operands)``: every operand was cut at the same leading-axis boundaries
    (`leading_splits` / `leading_block`), so the blocks are independent -- no collective."""
    from ._elemwise import elemwise

    return elemwise(func, *local_blocks, **kwargs)


def reduce_leading(x_local, method, axis=None, keepdims=False, group=None, **kwargs):
    """``x.reduce(method, axis)`` for an array range-partitioned on axis 0.

    Axis 0 kept: the local result IS this rank's block of the answer (no collective).  Axis 0 reduced: every rank
    reduces its block to a sparse partial over the kept axes, the partials' (key, value) streams are all-gathered
    (variable length) and stacked on a new leading axis of extent `world`, and one more device reduction over that
    axis combines them -- the same result on every rank.  Requires a fill value that the reduction leaves unchanged
    (0 for add, 0/1 for multiply, anything for max/min/and/or), the only case in which partial fill values agree."""
    from ._coo import COO
    from ._utils import equivalent, normalize_axis

    dist = _dist()
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    ax = normalize_axis(axis, x_local.ndim)
    ax = tuple(range(x_local.ndim)) if ax is None or ax == (None,) else (ax if isinstance(ax, tuple) else (ax,))
    if 0 not in ax or world == 1:
        return x_local.reduce(method, axis=ax, keepdims=keepdims, **kwargs)
    part = x_local.reduce(method, axis=ax, keepdims=False, **kwargs)
    t = D.torch()
    kept = tuple(part.shape)
    size = int(np.prod(kept)) if kept else 1
    if not kept:
        # full reduction: the partial is one dense element (its own fill value); combine the `world` elements
        keys = Kn.full(1, 0, np.int64)
        vals = D.upload(np.asarray(part.todense()).reshape(1))
        part_fill = vals.new_zeros(1)[0].item()
    else:
        if not equivalent(part.fill_value, part.dtype.type(x_local.fill_value)):
            raise ValueError("reduce_leading: the reduction changes the fill value, so row-block partials cannot be "
                             "combined; gather the operand instead")
        part_fill = part.fill_value
        c = part if isinstance(part, COO) else part.tocoo()
        if c.nnz:
            keys, vals = c.sorted_keys(), c._data_dev()
        else:
            keys, vals = Kn.full(0, 0, np.int64), Kn.full(0, 0, part.dtype)
    all_keys = all_gather_varlen(keys, group)
    all_vals = all_gather_varlen(vals, group)
    stacked_keys = t.cat([k + r * size for r, k in enumerate(all_keys)])
    stacked = COO._from_device(None, t.cat(all_vals), (world,) + kept, part_fill, keys=stacked_keys) \
        if int(stacked_keys.shape[0]) else COO(np.zeros((1 + len(kept), 0), dtype=np.intp),
                                               np.empty(0, dtype=part.dtype), shape=(world,) + kept,
                                               fill_value=part_fill)
    out = stacked.reduce(method, axis=(0,), **{k: v for k, v in kwargs.items() if k != "dtype"})
    if keepdims:
        shape = list(x_local.shape)
        for a in ax:
            shape[a] = 1
        out = out.reshape(tuple(shape)) if out.ndim or shape else out
    return out
