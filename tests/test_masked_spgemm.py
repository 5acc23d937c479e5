"""masked_matmul(s, a, b) == s * (a @ b) for sparse s, a, b (K10), against the reference's unfused expression.

The golden cases (tests/golden/masked_spgemm_api.npz, from tests/golden/make_masked_golden.py) run on the NumPy mock of
the kernel layer and on the B200 (`sp` fixture).  At the stored positions of `s` the result is bit-exact with upstream
(NaN payloads aside); where upstream stores nothing outside `s` it is equal outright.  The GPU-only tests at the end
judge sizes the reference cannot run against the unfused device path, SciPy and the C restatement of upstream's
product kernel."""
import numpy as np
import pytest
import torch

from _api import sp  # noqa: F401  (fixture)
from _golden import cases as golden_cases
from _masked_oracle import masked_ref_csr, masked_spgemm_np, same_bits_nan

CASES = golden_cases("masked_spgemm_api")
_PAIRS = {("float32", "float32"), ("float32", "float64"), ("float64", "float64"), ("int64", "int64"),
          ("int64", "float64"), ("bool", "bool"), ("bool", "int64"), ("bool", "float32"), ("bool", "float64")}


@pytest.fixture
def msp(sp, monkeypatch):  # noqa: F811
    """`sp`, plus (on the mock backend) a NumPy restatement of the K10 wrapper with the kernel's argument contract."""
    from sparse_b200 import _device as D
    from sparse_b200 import _kernels as Kn

    if D._TEST_CPU:
        def masked_spgemm(s_indptr, s_cols, s_vals, a_indptr, a_indices, a_data, bt_indptr, bt_indices, bt_data,
                          M, N, K):
            idx = (s_indptr, s_cols, a_indptr, a_indices, bt_indptr, bt_indices)
            assert all(x.dtype == s_indptr.dtype for x in idx) and s_indptr.dtype in (torch.int32, torch.int64)
            assert a_data.dtype == bt_data.dtype
            pair = (str(a_data.numpy().dtype), str(s_vals.numpy().dtype))
            assert pair in _PAIRS, f"dtype pair {pair} outside the kernel's list"
            for x, rows in ((a_indices, a_indptr), (bt_indices, bt_indptr)):  # the kernel needs sorted rows
                xi, ri = x.numpy().astype(np.int64), rows.numpy().astype(np.int64)
                assert all((np.diff(xi[ri[r]:ri[r + 1]]) > 0).all() for r in range(len(ri) - 1))
            out = masked_spgemm_np(*(t.numpy() for t in (s_indptr, s_cols, s_vals, a_indptr, a_indices, a_data,
                                                          bt_indptr, bt_indices, bt_data)), M, N, K)
            return torch.from_numpy(np.ascontiguousarray(out))

        monkeypatch.setattr(Kn, "masked_spgemm", masked_spgemm)
    yield sp


def operand(sp, case, prefix, fmt):  # noqa: F811
    a = case.sub(prefix)
    shape = tuple(int(x) for x in a["shape"])
    if fmt == "raw":  # unsorted rows, stored as the earlier product left them
        assert str(a["kind"]) == "gcxs"
        return sp.GCXS((a["data"], a["indices"], a["indptr"]), shape=shape,
                       compressed_axes=tuple(int(c) for c in a["ca"]))
    x = sp.COO(np.array(a["coords"]), np.array(a["data"]), shape=shape, has_duplicates=False, sorted=True)
    if fmt == "coo":
        return x
    return x.asformat("gcxs", compressed_axes=(0,) if fmt == "csr" else (1,))


def operands(sp, case):  # noqa: F811
    return (operand(sp, case, "s_", case["fs"]), operand(sp, case, "a_", case["fa"]),
            operand(sp, case, "b_", case["fb"]))


def check_against(sp, got, case, prefix):  # noqa: F811
    w = case.sub(prefix)
    assert tuple(got.shape) == tuple(int(x) for x in w["shape"])
    fill = w["fill"][()]
    assert got.fill_value.dtype == fill.dtype and same_bits_nan(np.asarray(got.fill_value), np.asarray(fill))
    assert got.dtype == w["data"].dtype, (got.dtype, w["data"].dtype)
    if str(w["kind"]) == "coo":
        assert isinstance(got, sp.COO), type(got)
        assert np.array_equal(got.coords, w["coords"]), "coords differ"
    else:
        assert isinstance(got, sp.GCXS), type(got)
        assert got.compressed_axes == tuple(int(c) for c in w["ca"])
        assert np.array_equal(got.indices, w["indices"]), "indices differ"
        assert np.array_equal(got.indptr, w["indptr"]), "indptr differ"
        assert got.indices.dtype == w["indices"].dtype, (got.indices.dtype, w["indices"].dtype)
    assert same_bits_nan(got.data, w["data"]), "data not bit-identical"


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_golden_at_mask_positions(msp, case):
    s, a, b = operands(msp, case)
    got = msp.masked_matmul(s, a, b)
    check_against(msp, got, case, "r_")
    if case["outright"]:
        check_against(msp, got, case, "out_")


def test_golden_grid_covers_the_contract():
    names = [c["name"] for c in CASES]
    assert sum(n.startswith("fmt-") for n in names) == 27
    assert any(not c["outright"] for c in CASES), "a case where upstream stores entries outside s"
    assert sum(c["outright"] for c in CASES) >= 30, "cases where the two expressions agree outright"


TRI = [c for c in CASES if "triangles" in c]


@pytest.mark.parametrize("case", TRI, ids=[c["name"] for c in TRI])
def test_triangle_counts(msp, case):
    g = operand(msp, case, "s_", case["fs"])
    tot = msp.masked_matmul(g, g, g).sum()
    got = np.asarray(tot.todense() if hasattr(tot, "todense") else tot)[()]
    txt = case["triangles"]  # repr of a Python int or float
    want = int(txt) if txt.lstrip("-").isdigit() else float(txt)
    assert got == want and float(got).is_integer(), (got, want)


# ---- errors and the dense delegation ----------------------------------------------------------------------------
def _small(sp, dtype=np.float64, shape=(4, 5), seed=0):  # noqa: F811
    return sp.random(shape, density=0.5, random_state=np.random.default_rng(seed)).astype(dtype)


def test_nonzero_fill_value(msp):
    s, a, b = _small(msp, shape=(4, 5)), _small(msp, shape=(4, 3)), _small(msp, shape=(3, 5))
    a1 = msp.COO(a.coords, a.data, shape=a.shape, fill_value=1.0)
    with pytest.raises(ValueError, match="zero fill values"):
        msp.masked_matmul(s, a1, b)


def test_shape_mismatch(msp):
    s, a, b = _small(msp, shape=(4, 5)), _small(msp, shape=(4, 3)), _small(msp, shape=(2, 5))
    with pytest.raises(ValueError, match=r"s\(4, 5\), a\(4, 3\), b\(2, 5\)"):
        msp.masked_matmul(s, a, b)
    with pytest.raises(ValueError):
        msp.masked_matmul(_small(msp, shape=(3, 5)), _small(msp, shape=(4, 3)), _small(msp, shape=(3, 5)))


def test_sparse_dense_mix_is_a_type_error(msp):
    s, a, b = _small(msp, shape=(4, 5)), _small(msp, shape=(4, 3)), _small(msp, shape=(3, 5))
    for args in ((s, a, b.todense()), (s, a.todense(), b), (s.todense(), a, b)):
        with pytest.raises(TypeError, match="sddmm"):
            msp.masked_matmul(*args)


def test_complex_is_a_type_error(msp):
    s, a, b = _small(msp, shape=(4, 5)), _small(msp, shape=(4, 3)), _small(msp, shape=(3, 5))
    with pytest.raises(TypeError, match="complex"):
        msp.masked_matmul(s, a.astype(np.complex128), b)


def test_dense_operands_reach_sddmm(msp, monkeypatch):
    from sparse_b200 import _fused

    s = _small(msp, shape=(6, 7))
    rng = np.random.default_rng(1)
    a, b = rng.random((6, 3)), rng.random((3, 7))
    calls = []
    real = _fused.sddmm

    def spy(*args, **kwargs):
        calls.append(args)
        return real(*args, **kwargs)

    monkeypatch.setattr(_fused, "sddmm", spy)
    got = msp.masked_matmul(s, a, b)
    assert len(calls) == 1 and calls[0][0] is s and calls[0][1] is a and calls[0][2] is b
    want = real(s, a, b)
    assert type(got) is type(want) and np.array_equal(got.coords, want.coords)
    assert same_bits_nan(got.data, want.data)


def test_not_in_all(msp):
    assert "masked_matmul" not in msp.__all__ and callable(msp.masked_matmul)


# ---- B200 only: sizes the reference cannot run ------------------------------------------------------------------
def _sym_graph(rng, n, deg):
    import scipy.sparse as ss

    m = n * deg // 2
    r, c = rng.integers(0, n, m), rng.integers(0, n, m)
    keep = r != c
    g = ss.coo_matrix((np.ones(int(keep.sum())), (r[keep], c[keep])), shape=(n, n)).tocsr()
    g = ((g + g.T) > 0).astype(np.float32).tocsr()
    g.sort_indices()
    return g


def _chung_lu(rng, n, nnz, hubs, hub_deg):
    """Power-law expected degrees (exponent ~2.1) plus a few hubs; symmetric, sorted CSR, random values in [0.5, 1.5)."""
    import scipy.sparse as ss

    w = (np.arange(1, n + 1) ** (-1 / 1.1))
    w *= nnz / w.sum()
    w[:hubs] = hub_deg
    p = w / w.sum()
    m = int(w.sum() / 2)
    r, c = rng.choice(n, m, p=p), rng.choice(n, m, p=p)
    keep = r != c
    g = ss.coo_matrix((np.ones(int(keep.sum())), (r[keep], c[keep])), shape=(n, n)).tocsr()
    g = ((g + g.T) > 0).astype(np.float32).tocsr()
    g.sort_indices()
    g.data = (rng.random(g.nnz) + 0.5).astype(np.float32)
    return g


def _gcxs(sp, g):  # noqa: F811
    return sp.GCXS((g.data, g.indices.astype(np.int64), g.indptr.astype(np.int64)), shape=g.shape,
                   compressed_axes=(0,))


@pytest.mark.gpu
def test_gpu_graph_matches_unfused_and_scipy(sp):  # noqa: F811
    rng = np.random.default_rng(2026)
    n = 200_000
    g = _sym_graph(rng, n, 32)
    A = _gcxs(sp, g)
    fused = sp.masked_matmul(A, A, A)
    unfused = A @ A * A
    assert isinstance(fused, sp.GCXS) and fused.compressed_axes == unfused.compressed_axes
    fc, uc = fused.tocoo(), unfused.tocoo()
    fk = fc.coords[0] * n + fc.coords[1]
    uk = uc.coords[0] * n + uc.coords[1]
    # restricted to s's positions (here: every position upstream stores, since 0/1 products are never negative)
    keep = np.isin(uk, fk)
    assert keep.all()
    assert np.array_equal(fk, uk[keep]) and same_bits_nan(fc.data, uc.data[keep])
    tri = 0.0
    for r0 in range(0, n, 20_000):  # SciPy's (A @ A).multiply(A).sum() in row blocks (bounded host memory)
        blk = g[r0:r0 + 20_000]
        tri += float((blk @ g).multiply(blk).sum())
    tot = fused.sum()
    got = float(np.asarray(tot.todense() if hasattr(tot, "todense") else tot)[()])
    assert got == tri, (got, tri)


@pytest.mark.gpu
def test_gpu_power_law_hub_rows_against_oracle(sp):  # noqa: F811
    rng = np.random.default_rng(7)
    n = 20_000
    g = _chung_lu(rng, n, 300_000, hubs=4, hub_deg=3_000)
    assert np.diff(g.indptr).max() > 512  # longer than the kernel's shared-memory stage
    b = g.copy()
    b.data = (rng.random(b.nnz) * 2 - 1).astype(np.float32)
    s = g.copy()
    s.data = (rng.random(s.nnz) * 4 - 2).astype(np.float32)
    got = sp.masked_matmul(_gcxs(sp, s), _gcxs(sp, g), _gcxs(sp, b)).tocoo()
    want = masked_ref_csr((n, n), s.indptr, s.indices, s.data, g.indptr, g.indices, g.data, b.indptr, b.indices,
                          b.data, n)
    rows = np.repeat(np.arange(n), np.diff(s.indptr))
    keep = want.view(np.uint32) != 0  # +0 is dropped
    assert np.array_equal(got.coords[0], rows[keep]) and np.array_equal(got.coords[1], s.indices[keep])
    assert same_bits_nan(got.data, want[keep])


@pytest.mark.gpu
def test_gpu_unsorted_rows_against_oracle(sp):  # noqa: F811
    import scipy.sparse as ss

    rng = np.random.default_rng(11)
    n, k = 3_000, 400

    def rnd(shape, density):
        x = ss.random(*shape, density=density, random_state=rng, format="csr", dtype=np.float64)
        x.data = x.data * 2 - 1
        return _gcxs(sp, x)

    a = rnd((n, k), 0.02) @ rnd((k, n), 0.01)  # K4's row order: reverse first touch
    b = rnd((n, k), 0.02) @ rnd((k, n), 0.01)
    assert not all((np.diff(a.indices[a.indptr[r]:a.indptr[r + 1]]) > 0).all() for r in range(n))
    s = rnd((n, n), 0.01)
    got = sp.masked_matmul(s, a, b)
    bs = b.asformat("gcxs", compressed_axes=(0,))
    want = masked_ref_csr((n, n), s.indptr, s.indices, s.data, a.indptr, a.indices, a.data, bs.indptr, bs.indices,
                          bs.data, n)
    keep = want.view(np.uint64) != 0
    assert isinstance(got, sp.GCXS) and got.compressed_axes == (0,)
    rows = np.repeat(np.arange(n), np.diff(s.indptr))
    gc = got.tocoo()
    assert np.array_equal(gc.coords[0], rows[keep]) and np.array_equal(gc.coords[1], s.indices[keep])
    assert same_bits_nan(gc.data, want[keep])


@pytest.mark.gpu
def test_gpu_int64_indices_against_contract(sp):  # noqa: F811
    """The int64-index instantiations of K10 (taken when an extent or nnz exceeds int32), called through the wrapper on
    a power-law graph with hub rows longer than the stage: equal to the NumPy restatement and to the int32 run."""
    from sparse_b200 import _device as D
    from sparse_b200 import _kernels as Kn

    rng = np.random.default_rng(5)
    n = 8_000
    g = _chung_lu(rng, n, 80_000, hubs=3, hub_deg=1_500)
    assert np.diff(g.indptr).max() > 512
    bt = g.copy()
    bt.data = (rng.random(bt.nnz) * 2 - 1).astype(np.float32)  # rows of Bt = columns of b (sorted)
    s = g.copy()
    s.data = (rng.random(s.nnz) * 4 - 2).astype(np.float32)
    want = masked_spgemm_np(s.indptr, s.indices, s.data, g.indptr, g.indices, g.data, bt.indptr, bt.indices, bt.data,
                            n, n, n)
    for idt in (np.int64, np.int32):
        up = [D.upload(np.ascontiguousarray(x, dtype=idt)) for x in (s.indptr, s.indices, g.indptr, g.indices,
                                                                    bt.indptr, bt.indices)]
        out = Kn.masked_spgemm(up[0], up[1], D.upload(s.data), up[2], up[3], D.upload(g.data), up[4], up[5],
                               D.upload(bt.data), n, n, n)
        assert same_bits_nan(D.download(out), want), idt
