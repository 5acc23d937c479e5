"""masked_matmul_rowblock at world size 2 (`gloo`, NumPy mock of the kernel layer): each rank holds a block of rows of
`s` and `a` and a block of rows of `b`; the concatenated row blocks must equal the single-process result."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))


def _worker(rank, world, port, q):
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.dirname(HERE))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import _mock_kernels
        from _masked_oracle import masked_spgemm_np, same_bits_nan

        _mock_kernels.install()
        import sparse_b200 as sp
        from sparse_b200 import _dist as DD
        from sparse_b200 import _kernels as Kn

        def mock(*args):
            return torch.from_numpy(np.ascontiguousarray(masked_spgemm_np(*(t.numpy() for t in args[:9]), *args[9:])))

        Kn.masked_spgemm = mock
        rng = np.random.default_rng(31)  # same inputs on every rank
        M, K, N = 50, 40, 45

        def rnd(shape, density):
            x = sp.random(shape, density=density, random_state=rng).astype(np.float64)
            x = sp.COO(x.coords, (x.data * 2 - 1), shape=shape)
            return x.asformat("gcxs", compressed_axes=(0,))

        s, a, b = rnd((M, N), 0.3), rnd((M, K), 0.2), rnd((K, N), 0.2)
        want = sp.masked_matmul(s, a, b)
        rb = DD.nnz_balanced_splits(s.indptr, world)
        kb = DD.nnz_balanced_splits(b.indptr, world)
        r0, r1 = rb[rank], rb[rank + 1]
        k0, k1 = kb[rank], kb[rank + 1]
        s_local = sp.GCXS(DD.row_block(s.data, s.indices, s.indptr, r0, r1), shape=(r1 - r0, N), compressed_axes=(0,))
        a_local = sp.GCXS(DD.row_block(a.data, a.indices, a.indptr, r0, r1), shape=(r1 - r0, K), compressed_axes=(0,))
        b_local = sp.GCXS(DD.row_block(b.data, b.indices, b.indptr, k0, k1), shape=(k1 - k0, N), compressed_axes=(0,))
        got = DD.masked_matmul_rowblock(s_local, a_local, b_local)
        blocks = [None] * world
        dist.all_gather_object(blocks, (np.asarray(got.data), np.asarray(got.indices), np.asarray(got.indptr)))
        data = np.concatenate([blk[0] for blk in blocks])
        indices = np.concatenate([blk[1] for blk in blocks])
        ptrs, base = [np.zeros(1, np.int64)], 0
        for blk in blocks:
            ptrs.append(np.asarray(blk[2][1:], dtype=np.int64) + base)
            base += len(blk[0])
        indptr = np.concatenate(ptrs)
        ok = (isinstance(got, sp.GCXS) and got.compressed_axes == (0,) and np.array_equal(indptr, want.indptr)
              and np.array_equal(indices, want.indices) and same_bits_nan(data, want.data) and want.nnz > 0)
        q.put((rank, bool(ok)))
    finally:
        dist.destroy_process_group()


def test_masked_matmul_rowblock_world2():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 33500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=240) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, ok in res:
        assert ok, f"rank {rank}: masked_matmul_rowblock differs from the single-process result"
