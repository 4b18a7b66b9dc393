"""lcpm on sparse read-count matrices (scipy CSR / CSC / COO on the host, torch sparse CSR / COO on the device):
the counts are never expanded to genes x cells, and the result is bit for bit what the dense path gives on the same
counts (``toarray()`` / ``to_dense()``), for every option and row-block chunking."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

import normalisr_oracle as orc
from conftest import load_golden

pytestmark = pytest.mark.gpu

CHUNKINGS = ((1 << 30, 1 << 35), (8 * 300 * 50, 1 << 35), (8 * 300 * 50, 0))


def _same(a, b):
    """Two lcpm results (4-tuples of arrays / tensors / None) are identical, bit for bit."""
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert (x is None) == (y is None)
        if x is None:
            continue
        if isinstance(x, torch.Tensor):
            assert isinstance(y, torch.Tensor) and x.is_cuda and y.is_cuda
            assert x.dtype == y.dtype and torch.equal(x, y)
        else:
            assert isinstance(x, np.ndarray) and isinstance(y, np.ndarray)
            assert x.dtype == y.dtype and np.array_equal(x, y)


def _scipy_forms(dense):
    coo = sp.coo_matrix(dense)
    return {"csr": coo.tocsr(), "csc": coo.tocsc(), "coo": coo}


def _torch_forms(dense):
    t = torch.from_numpy(np.ascontiguousarray(dense)).cuda()
    return {"csr": t.to_sparse_csr(), "csc": t.to_sparse_csc(), "coo": t.to_sparse()}


@pytest.fixture
def norm():
    from normalisr_b200 import normalisr
    return normalisr


@pytest.fixture
def lc():
    from normalisr_b200 import lcpm
    return lcpm


@pytest.fixture
def counts():
    return load_golden("lcpm_counts")


@pytest.fixture
def resample():
    return load_golden("lcpm_resample")


def test_golden_host_formats_and_chunkings(norm, lc, counts, monkeypatch):
    g = counts
    for chunk, hold in CHUNKINGS:
        monkeypatch.setattr(lc, "_ROW_CHUNK_BYTES", chunk)
        monkeypatch.setattr(lc, "_HOLD_BYTES", hold)
        want = norm.lcpm(g["reads"])
        np.testing.assert_allclose(want[0], g["lcpm"], rtol=1e-12, atol=1e-12)
        for name, m in _scipy_forms(g["reads"]).items():
            got = norm.lcpm(m)
            _same(got, want)
            np.testing.assert_allclose(got[3], g["cov"], rtol=1e-13)
        m = _scipy_forms(g["reads"])["csr"]
        _same(norm.lcpm(m, lowmem=False, nocov=True), norm.lcpm(g["reads"], lowmem=False, nocov=True))
        _same(norm.lcpm(m, normalize=False, ntot=10 ** 9), norm.lcpm(g["reads"], normalize=False, ntot=10 ** 9))
    out = norm.lcpm(_scipy_forms(g["reads"].astype(np.int32))["csc"], lowmem=False, nocov=True)
    np.testing.assert_allclose(out[1], g["mean"], rtol=1e-12, atol=1e-12)
    assert (out[2] == 0).all() and out[3] is None
    out = norm.lcpm(_scipy_forms(g["reads"])["coo"], normalize=False, ntot=10 ** 9)
    np.testing.assert_allclose(out[0], g["lcpm_raw"], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(out[3], g["cov_raw"], rtol=1e-13)


def test_golden_device_formats(norm, counts):
    g = counts
    for name, t in _torch_forms(g["reads"].astype(np.int64)).items():
        dense = t.to_dense()
        for kw in ({}, {"lowmem": False, "nocov": True}, {"normalize": False, "ntot": 10 ** 9}):
            got = norm.lcpm(t, **kw)
            assert got[0].is_cuda
            _same(got, norm.lcpm(dense, **kw))
        np.testing.assert_allclose(norm.lcpm(t)[0].cpu().numpy(), g["lcpm"], rtol=1e-12, atol=1e-12)


def test_resampling_host_and_device(norm, lc, resample, monkeypatch):
    g = resample
    vs, seed = float(g["varscale"]), int(g["seed"])
    for chunk, hold in CHUNKINGS:
        monkeypatch.setattr(lc, "_ROW_CHUNK_BYTES", chunk)
        monkeypatch.setattr(lc, "_HOLD_BYTES", hold)
        for name, m in _scipy_forms(g["reads"]).items():
            for lowmem in (True, False):
                got = norm.lcpm(m, varscale=vs, seed=seed, lowmem=lowmem)
                _same(got, norm.lcpm(g["reads"], varscale=vs, seed=seed, lowmem=lowmem))
    got = norm.lcpm(_scipy_forms(g["reads"])["csr"], varscale=vs, seed=seed, lowmem=False)
    np.testing.assert_allclose(got[0], g["lcpm_full"], rtol=1e-11, atol=1e-11)
    np.testing.assert_allclose(got[1], g["mean_full"], rtol=1e-11, atol=1e-11)
    np.testing.assert_allclose(got[2], g["var_full"], rtol=1e-11, atol=1e-14)
    np.testing.assert_allclose(got[3], g["cov"], rtol=1e-13)
    for name, t in _torch_forms(g["reads"].astype(np.int64)).items():
        dense = t.to_dense()
        for kw in ({"lowmem": False}, {"normalize": False, "ntot": 10 ** 9}, {"nocov": True}):
            _same(norm.lcpm(t, varscale=0.7, seed=5, **kw), norm.lcpm(dense, varscale=0.7, seed=5, **kw))


def _random_counts(rng, genes, cells, density):
    dense = np.zeros((genes, cells), dtype=np.int64)
    mask = rng.random((genes, cells)) < density
    dense[mask] = rng.negative_binomial(1, 0.3, size=int(mask.sum())) + 1
    return dense


def test_larger_random_against_dense_and_oracle(norm):
    rng = np.random.default_rng(31)
    dense = _random_counts(rng, 3000, 20000, 0.05)
    dense[:, 0] += 1                                               # no empty cell
    dense[rng.choice(np.arange(6, 2999), 40, replace=False)] = 0   # genes without a stored entry
    dense[5, :50] = np.arange(4070, 4120)                          # counts at and beyond the 4,096-entry table
    dense[2999, 100:110] = 10 ** 6
    m = sp.csr_matrix(dense)
    want = norm.lcpm(dense)
    got = norm.lcpm(m)
    _same(got, want)
    ref = orc.lcpm(dense)
    np.testing.assert_allclose(got[0], ref[0], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(got[3], ref[3], rtol=1e-13)
    t = torch.from_numpy(dense).cuda().to_sparse_csr()
    _same(norm.lcpm(t), norm.lcpm(t.to_dense()))
    # every entry stored
    full = rng.integers(1, 50, size=(200, 3000))
    _same(norm.lcpm(sp.coo_matrix(full)), norm.lcpm(full))
    _same(norm.lcpm(sp.csr_matrix(full), lowmem=False), norm.lcpm(full, lowmem=False))


def test_counts_beyond_int32(norm):
    """Counts of 2^31 and more: the CSR kernels expand the tile as int64."""
    rng = np.random.default_rng(5)
    dense = _random_counts(rng, 150, 700, 0.1)
    dense[:, 3] += 1
    dense[7, 11] = 2 ** 31 + 5
    dense[140, 600] = 3 * 2 ** 32
    for m in _scipy_forms(dense).values():
        _same(norm.lcpm(m), norm.lcpm(dense))
    _same(norm.lcpm(sp.csr_matrix(dense), normalize=False, lowmem=False), norm.lcpm(dense, normalize=False, lowmem=False))
    t = torch.from_numpy(dense).cuda().to_sparse_csr()
    _same(norm.lcpm(t), norm.lcpm(t.to_dense()))


def _noncanonical(rng, genes, cells, nnz, dtype):
    """Entries in random order with duplicates and explicit zeros; every cell has reads."""
    r = rng.integers(0, genes, nnz)
    c = rng.integers(0, cells, nnz)
    v = rng.integers(0, 30, nnz).astype(np.float64)
    v[::17] = 0                                                     # explicit zeros
    r = np.concatenate([r, r[:50], np.arange(cells) % genes])      # duplicates of the first 50 entries
    c = np.concatenate([c, c[:50], np.arange(cells)])
    v = np.concatenate([v, v[:50], np.full(cells, 2.0)])
    if np.dtype(dtype).kind == 'f':
        v = v + 0.6                                                 # 0.6 + 0.6 crosses an integer
    return r, c, v.astype(dtype)


def _toarray_counts(m):
    d = m.toarray()
    return d if np.issubdtype(d.dtype, np.integer) else d.astype(np.int64)


def test_noncanonical_host_input(norm):
    rng = np.random.default_rng(8)
    genes, cells = 130, 900
    for dtype in (np.int32, np.int64, np.float32, np.float64, np.uint16):
        r, c, v = _noncanonical(rng, genes, cells, 6000, dtype)
        coo = sp.coo_matrix((v, (r, c)), shape=(genes, cells))
        # CSR with unsorted column indices and duplicates, int32 and int64 index arrays
        order = np.argsort(r, kind="stable")
        indptr = np.r_[0, np.cumsum(np.bincount(r, minlength=genes))]
        mats = [coo, coo.tocsc()]
        for it in (np.int32, np.int64):
            mats.append(sp.csr_matrix((v[order], c[order].astype(it), indptr.astype(it)), shape=(genes, cells)))
            mats.append(sp.coo_matrix((v, (r.astype(it), c.astype(it))), shape=(genes, cells)))
        for m in mats:
            want = norm.lcpm(_toarray_counts(m))
            before = [np.array(getattr(m, a), copy=True) for a in ("data", "indices", "indptr", "row", "col") if hasattr(m, a)]
            _same(norm.lcpm(m), want)
            _same(norm.lcpm(m, varscale=0.5, seed=3, lowmem=False), norm.lcpm(_toarray_counts(m), varscale=0.5, seed=3,
                                                                                 lowmem=False))
            after = [getattr(m, a) for a in ("data", "indices", "indptr", "row", "col") if hasattr(m, a)]
            for x, y in zip(before, after):
                assert x.dtype == y.dtype and np.array_equal(x, y)
    # float duplicates: 0.6 + 0.6 = 1.2 -> 1 (each alone would be 0)
    m = sp.coo_matrix((np.array([0.6, 0.6, 3.0, 2.0]), (np.array([0, 0, 1, 1]), np.array([1, 1, 0, 1]))), shape=(2, 2))
    assert _toarray_counts(m)[0, 1] == 1
    _same(norm.lcpm(m), norm.lcpm(_toarray_counts(m)))


def test_noncanonical_device_input(norm):
    rng = np.random.default_rng(9)
    genes, cells = 120, 1000
    for dtype in (torch.int32, torch.int64, torch.float64):
        r, c, v = _noncanonical(rng, genes, cells, 5000, np.int64)
        vv = torch.from_numpy(v).to(dtype)
        if dtype.is_floating_point:
            vv = vv + 0.5                                          # 0.5 + 0.5 is exact in any order
        ij = torch.from_numpy(np.stack([r, c]))
        t = torch.sparse_coo_tensor(ij, vv, (genes, cells)).cuda()    # uncoalesced: duplicates and any order
        assert not t.is_coalesced()
        vals0, idx0 = t._values().clone(), t._indices().clone()
        _same(norm.lcpm(t), norm.lcpm(t.to_dense()))
        _same(norm.lcpm(t, varscale=0.3, seed=2, lowmem=False), norm.lcpm(t.to_dense(), varscale=0.3, seed=2, lowmem=False))
        assert torch.equal(t._values(), vals0) and torch.equal(t._indices(), idx0)
        # CSR with column indices descending within rows (no duplicates)
        key, first = np.unique(r * cells + c, return_index=True)
        ru, cu = key // cells, key % cells
        order = np.lexsort((-cu, ru))
        crow = torch.from_numpy(np.r_[0, np.cumsum(np.bincount(ru, minlength=genes))])
        tc = torch.sparse_csr_tensor(crow, torch.from_numpy(cu[order]), vv[torch.from_numpy(first[order])],
                                     (genes, cells)).cuda()
        _same(norm.lcpm(tc), norm.lcpm(tc.to_dense()))


def test_errors_match_dense_path(norm):
    with pytest.raises(ValueError):
        norm.lcpm(sp.csr_matrix(np.array([[1, 0, -2], [3, 4, 1]])))                 # negative count
    with pytest.raises(ValueError):
        norm.lcpm(sp.csr_matrix(np.array([[1, -1, 2], [3, 4, 1]])), varscale=0.5)
    with pytest.raises(ValueError):
        norm.lcpm(sp.csr_matrix(np.array([[1, 0, 2], [3, 0, 1]])))                  # a cell with no reads
    with pytest.raises(AssertionError):
        norm.lcpm(sp.csr_matrix((3, 4), dtype=np.int64))                             # no reads at all
    with pytest.raises(AssertionError):
        norm.lcpm(sp.coo_matrix((np.zeros(3), ([0, 1, 2], [0, 1, 3])), shape=(3, 4)))  # explicit zeros only
    for bad in (np.nan, np.inf, -np.inf):
        with pytest.raises(ValueError):
            norm.lcpm(sp.csr_matrix(np.array([[1.0, 2.0, bad], [3.0, 4.0, 1.0]])))
        with pytest.raises(ValueError):
            norm.lcpm(torch.tensor([[1.0, 2.0, bad], [3.0, 4.0, 1.0]], device="cuda").to_sparse_csr())
    with pytest.raises(ValueError):
        norm.lcpm(torch.tensor([[1, 0, -2], [3, 4, 1]], device="cuda").to_sparse())
    with pytest.raises(ValueError):
        norm.lcpm(torch.ones(4, dtype=torch.int64, device="cuda").to_sparse())      # wrong ndim
    with pytest.raises(ValueError):
        norm.lcpm(sp.csr_matrix(np.ones((3, 4), dtype=int)), varscale=-1)


def test_no_densification_on_the_host(norm, counts, monkeypatch):
    def refuse(self, *a, **k):
        raise AssertionError("densified on the host")
    want = norm.lcpm(counts["reads"])
    for name, m in _scipy_forms(counts["reads"]).items():
        for attr in ("toarray", "todense"):
            monkeypatch.setattr(type(m), attr, refuse)
        _same(norm.lcpm(m), want)


def test_no_densification_on_the_device(norm):
    rng = np.random.default_rng(4)
    genes, cells = 2000, 20000
    dense = _random_counts(rng, genes, cells, 0.05)
    dense[:, 0] += 1
    t = torch.from_numpy(dense).cuda().to_sparse_csr()
    del dense
    sparse_bytes = sum(x.numel() * x.element_size() for x in (t.crow_indices(), t.col_indices(), t.values()))
    out_bytes = 8 * genes * cells
    norm.lcpm(t)                                                   # tables, scratch and the allocator warmed up
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out = norm.lcpm(t)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    assert peak < out_bytes + sparse_bytes + (16 << 20), (peak, out_bytes, sparse_bytes)
    assert peak < out_bytes + 4 * genes * cells                    # well under a dense int32 copy of the counts
    assert out[0].shape == (genes, cells)
