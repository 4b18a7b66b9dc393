"""The co-expression network in one call (``coexnet``) and the binary network in CSR form
(``binnet(..., sparse=True)``; csrc/binnet.cu ``nsr_binnet_count`` + ``nsr_binnet_csr_fill``).
CPU: the host-side assembly of CSR pieces, the oracle's network in CSR form against the golden nets, the C ABI,
and the new kernels' register use.  GPU: CSR structure equal to ``csr_matrix`` of the dense network bit for bit,
and ``coexnet`` equal to ``binnet(coex(...)[0])`` on one GPU and on several."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import scipy.sparse
import torch

import normalisr_oracle as orc
from conftest import ROOT, load_golden

gpu = pytest.mark.gpu


def _golden_nets(name):
    g = load_golden(name)
    P = g["P"]
    nets = [np.unpackbits(g["net"][k], axis=1)[:, :P.shape[1]].astype(bool) for k in range(len(g["qcut"]))]
    return P, g["qcut"], nets


def _same_csr(got, want):
    """Same CSR arrays (index dtype included) and all-True bool data."""
    want = scipy.sparse.csr_matrix(want)
    assert isinstance(got, scipy.sparse.csr_matrix) and got.shape == want.shape
    assert got.indptr.dtype == want.indptr.dtype and got.indices.dtype == want.indices.dtype
    assert np.array_equal(got.indptr, want.indptr) and np.array_equal(got.indices, want.indices)
    assert got.data.dtype == np.bool_ and got.data.all() and got.data.size == want.nnz


def _same_torch_csr(got, want):
    want = scipy.sparse.csr_matrix(want)
    assert got.is_cuda and got.layout == torch.sparse_csr and got.dtype == torch.bool
    assert tuple(got.shape) == want.shape
    crow, col = got.crow_indices().cpu().numpy(), got.col_indices().cpu().numpy()
    assert crow.dtype == want.indptr.dtype and col.dtype == want.indices.dtype
    assert np.array_equal(crow, want.indptr) and np.array_equal(col, want.indices)
    assert bool(got.values().all()) and got.values().numel() == want.nnz


# --------------------------------------------------------------------------------------------------- CPU
def test_concat_csr_pieces_with_empty_rows_and_blocks():
    """Per-device (or per-chunk) CSR pieces -> one CSR structure: pieces with empty rows, empty pieces (a GPU
    without rows), pieces whose row pointers do not start at 0, and the values carried along."""
    from normalisr_b200.binnet import concat_csr
    rng = np.random.default_rng(4)
    n = 300
    for trial in range(20):
        dense = rng.random((n, n)) < rng.choice([0.0, 0.01, 0.2])
        dense[rng.random(n) < 0.3] = False                           # empty rows
        vals = rng.random((n, n))
        cuts = np.unique(np.concatenate([[0, n], rng.integers(0, n, size=rng.integers(0, 6))]))
        pieces = []
        for a, b in zip(cuts[:-1], cuts[1:]):
            m = scipy.sparse.csr_matrix(dense[a:b])
            off = int(rng.integers(0, 1000))
            pieces.append((m.indptr.astype(np.int64) + off, m.indices, vals[a:b][dense[a:b]]))
            if trial % 3 == 0:
                pieces.append((np.full(1, 7, np.int64), np.zeros(0, np.int32), np.zeros(0)))    # a block of 0 rows
        indptr, indices, v = concat_csr(pieces, n)
        want = scipy.sparse.csr_matrix(dense)
        assert indptr.dtype == np.int32 and indices.dtype == np.int32
        assert np.array_equal(indptr, want.indptr) and np.array_equal(indices, want.indices)
        assert np.array_equal(v, vals[dense])


def test_concat_csr_switches_to_int64():
    """int32 while the entry count and the size fit, int64 (both arrays) beyond - the rule of scipy and torch."""
    from normalisr_b200.binnet import concat_csr, index_dtype
    assert index_dtype(2 ** 31 - 1, 10) == np.int32 and index_dtype(2 ** 31, 10) == np.int64
    assert index_dtype(5, 2 ** 31) == np.int64
    pieces = [(np.array([0, 2]), np.array([1, 3], np.int32)), (np.array([0, 1]), np.array([0], np.int32))]
    indptr, indices = concat_csr(pieces, 2 ** 31)
    assert indptr.dtype == np.int64 and indices.dtype == np.int64
    assert np.array_equal(indptr, [0, 2, 3]) and np.array_equal(indices, [1, 3, 0])


@pytest.mark.parametrize("name", ["binnet_coex", "binnet_ties"])
def test_oracle_net_in_csr_form_matches_golden(name):
    P, qcuts, nets = _golden_nets(name)
    for q, want in zip(qcuts, nets):
        if want.sum() == 0:
            with pytest.raises(RuntimeError):
                orc.binnet(P, q)
            continue
        _same_csr(scipy.sparse.csr_matrix(orc.binnet(P, q)), want)


def test_csr_entry_points_in_the_abi():
    from normalisr_b200 import _lib
    lib = _lib.load()
    for name in ("nsr_binnet_count", "nsr_binnet_csr_fill"):
        assert name in _lib.exported_symbols() and getattr(lib, name).argtypes
    header = open(os.path.join(ROOT, "include", "normalisr_b200.h")).read()
    assert "int nsr_binnet_count(" in header and "int nsr_binnet_csr_fill(" in header


@pytest.mark.skipif(shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"),
                    reason="needs nvcc")
def test_binnet_kernels_do_not_spill(tmp_path):
    """Every kernel of csrc/binnet.cu - the dense row kernels, their count variants and the CSR fill - compiles
    for sm_100a without local-memory spills."""
    from normalisr_b200 import _build
    res = subprocess.run([_build._nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17",
                          "-Xptxas", "-v", "-c", "-o", str(tmp_path / "binnet.o"),
                          os.path.join(_build.CSRC, "binnet.cu")], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-2000:]
    entries = re.findall(r"Compiling entry function '(\w+)'", res.stderr)
    spills = re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", res.stderr)
    assert len(entries) == 8 and len(spills) == 8
    assert any("csr_fill_kernelIiE" in e for e in entries) and any("csr_fill_kernelIlE" in e for e in entries)
    assert all(s == ("0", "0") for s in spills), spills


# --------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(params=["keys", "values"])
def row_kernel(request):
    """Both row kernels of csrc/binnet.cu (``binnet_keys`` 1 / 0)."""
    from normalisr_b200 import engine
    engine.set_option("binnet_keys", 1 if request.param == "keys" else 0)
    yield request.param
    engine.set_option("binnet_keys", 1)


@gpu
@pytest.mark.parametrize("name", ["binnet_coex", "binnet_ties"])
def test_sparse_binnet_golden(name, row_kernel, monkeypatch):
    """Every golden cutoff, host input (in one chunk and in many) and CUDA input."""
    from normalisr_b200 import binnet as bn, normalisr as norm
    P, qcuts, nets = _golden_nets(name)
    Pd = torch.from_numpy(P).cuda()
    for chunk_rows in (None, 7):
        if chunk_rows:
            monkeypatch.setattr(bn, "_ROW_CHUNK_BYTES", 8 * P.shape[0] * chunk_rows)
        for q, want in zip(qcuts, nets):
            if want.sum() == 0:
                for x in (P, Pd):
                    with pytest.raises(RuntimeError):
                        norm.binnet(x, q, sparse=True)
                continue
            _same_csr(norm.binnet(P, q, sparse=True), want)
            _same_torch_csr(norm.binnet(Pd, q, sparse=True), want)


def _csr_of_rows(ctx, Pm, q, diag0):
    """(dense uint8 rows, indptr, indices, P_e, D_e) of the same rows through both paths."""
    from normalisr_b200 import binnet as bn
    dense, _ = bn.binnet_rows(ctx, Pm, q, diag0)
    D = Pm * 3.0 - 1.0
    indptr, indices, p_e, d_e = bn.csr_rows(ctx, Pm, q, diag0, D=D)
    return (dense.cpu().numpy().astype(bool), indptr.cpu().numpy(), indices.cpu().numpy(), p_e.cpu().numpy(),
            d_e.cpu().numpy(), D.cpu().numpy())


@gpu
def test_sparse_rows_wide_offset_diagonal_and_ties(row_kernel):
    """The shapes of the dense row tests: rows wider than shared memory (the L2 re-read kernel), diagonals at an
    offset or outside the block, odd widths, unaligned rows, tied and slowly converging rows (window overflow ->
    fallback), negative zero.  CSR equals csr_matrix of the dense rows; P_e / D_e are the values at the edges."""
    from normalisr_b200 import engine
    rng = np.random.default_rng(9)
    ctx = engine.context(0)
    cases = []
    for cols, diag0 in ((30011, 0), (30011, 29990), (30011, -5), (5000, 4990), (4999, 3), (25000, 7), (50001, 49000),
                        (100003, 5)):
        cases.append((torch.from_numpy(rng.random((12, cols)) ** rng.integers(1, 8, size=(12, 1))).cuda(), diag0))
    cols = 6000
    k = np.arange(1, cols + 1)
    tied = [0.1 * k / cols * (1 - 1e-9 * rng.random(cols)), 0.1 * k / cols * (1 + 1e-3 * rng.random(cols)),
            np.where(rng.random(cols) < 0.5, 0.0123456, rng.random(cols)), np.full(cols, 0.04),
            np.where(rng.random(cols) < 0.3, -0.0, rng.random(cols) ** 4), np.sort(rng.random(cols)) ** 2 * 0.2]
    cases.append((torch.from_numpy(np.array([rng.permutation(r) for r in tied])).cuda(), -cols - 10))
    buf = torch.zeros(6 * 4003 + 8, dtype=torch.float64, device="cuda")               # rows at odd offsets
    view = buf[1:1 + 6 * 4003].view(6, 4003)[:, :3999]
    view.copy_(cases[-1][0][:, :3999])
    cases.append((view, 2))
    for Pm, diag0 in cases:
        for q in (0.1, 0.05, 1e-3):
            dense, indptr, indices, p_e, d_e, D = _csr_of_rows(ctx, Pm, q, diag0)
            want = scipy.sparse.csr_matrix(dense)
            assert np.array_equal(indptr, want.indptr) and np.array_equal(indices, want.indices), (Pm.shape, q, diag0)
            rows = np.repeat(np.arange(dense.shape[0]), np.diff(indptr))
            Ph = Pm.cpu().numpy()
            assert np.array_equal(p_e, Ph[rows, indices]) and np.array_equal(d_e, D[rows, indices])


@gpu
def test_sparse_binnet_errors():
    from normalisr_b200 import normalisr as norm
    P = np.random.default_rng(1).random((50, 50))
    for x in (P, torch.from_numpy(P).cuda()):
        with pytest.raises(ValueError):
            norm.binnet(x[:, :40], 0.1, sparse=True)
        with pytest.raises(ValueError):
            norm.binnet(x[:1, :1], 0.1, sparse=True)
        for q in (0.0, 1.0, -1, 2):
            with pytest.raises(ValueError):
                norm.binnet(x, q, sparse=True)
        bad = x.clone() if isinstance(x, torch.Tensor) else x.copy()
        bad[3, 4] = np.nan
        with pytest.raises(AssertionError):
            norm.binnet(bad, 0.1, sparse=True)
        bad[3, 4] = 1.5
        with pytest.raises(AssertionError):
            norm.binnet(bad, 0.1, sparse=True)
    with pytest.raises(RuntimeError):
        norm.binnet(np.ones((20, 20)), 0.5, sparse=True)


@pytest.fixture(scope="module")
def problem():
    """1,900 genes (not a multiple of the 128-row tile) x 3,000 cells with planted modules."""
    from normalisr_b200 import synth
    p = synth.device_problem(1012, 1900, 3000, "cuda")
    return p["dt"].cpu().numpy(), p["dc"].cpu().numpy()


def _reference(dt, dc, q):
    """What coexnet must equal: coex on one GPU, then binnet."""
    from normalisr_b200 import normalisr as norm
    P, D, var = norm.coex(dt, dc)
    return P, D, var, norm.binnet(P, q)


def _check_coexnet(dt, dc, q, ref, **ka):
    from normalisr_b200 import normalisr as norm
    P, D, var, want = ref
    net, v = norm.coexnet(dt, dc, q, **ka)
    assert isinstance(net, np.ndarray) and net.dtype == np.bool_ and np.array_equal(net, want)
    assert np.array_equal(v, var)
    net, v, p_e, d_e = norm.coexnet(dt, dc, q, sparse=True, edge_values=True, **ka)
    _same_csr(net, want)
    assert np.array_equal(v, var)
    rows = np.repeat(np.arange(net.shape[0]), np.diff(net.indptr))
    assert np.array_equal(p_e, P[rows, net.indices]) and np.array_equal(d_e, D[rows, net.indices])
    net, v = norm.coexnet(dt, dc, q, sparse=True, **ka)
    _same_csr(net, want)


@gpu
def test_coexnet_one_gpu_host_and_device_input(problem):
    from normalisr_b200 import normalisr as norm
    dt, dc = problem
    for q in (0.05, 1e-4):
        ref = _reference(dt, dc, q)
        _check_coexnet(dt, dc, q, ref)
        P, D, var, want = ref
        dt_d, dc_d = torch.from_numpy(dt).cuda(), torch.from_numpy(dc).cuda()
        net, v = norm.coexnet(dt_d, dc_d, q)
        assert net.is_cuda and net.dtype == torch.bool and np.array_equal(net.cpu().numpy(), want)
        assert v.is_cuda and np.array_equal(v.cpu().numpy(), var)
        net, v, p_e, d_e = norm.coexnet(dt_d, dc_d, q, sparse=True, edge_values=True)
        _same_torch_csr(net, want)
        crow, col = net.crow_indices().cpu().numpy(), net.col_indices().cpu().numpy()
        rows = np.repeat(np.arange(net.shape[0]), np.diff(crow))
        assert np.array_equal(p_e.cpu().numpy(), P[rows, col]) and np.array_equal(d_e.cpu().numpy(), D[rows, col])
    with pytest.raises(ValueError):
        norm.coexnet(dt, dc, 0.05, edge_values=True)
    with pytest.raises(ValueError):
        norm.coexnet(dt, dc, 1.0)


@gpu
def test_coexnet_forced_cell_chunks(problem, monkeypatch):
    """The contraction in cell chunks (the k_chunk path, which rounds the float64 sum of the chunks differently
    from one pass): the same network and edge values as coex + binnet under the same chunking."""
    from normalisr_b200 import engine
    dt, dc = problem
    monkeypatch.setattr(engine, "plan_k_chunk", lambda *a, **k: 1024)
    _check_coexnet(dt, dc, 0.05, _reference(dt, dc, 0.05))


@gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs in one process")
def test_coexnet_all_devices_one_process(problem, monkeypatch):
    """Several GPUs from one process: every device ends up with complete rows of its block (block-pair
    transposes copied peer to peer) and thresholds them; bit-identical to one GPU in both forms, with even and
    uneven row blocks, and with the contraction redone in cell chunks."""
    from normalisr_b200 import engine
    dt, dc = problem
    ref = _reference(dt, dc, 0.05)
    lists = ["all"] + ([[0, 1, 2]] if torch.cuda.device_count() >= 3 else []) + [[1, 0]]
    for devices in lists:
        _check_coexnet(dt, dc, 0.05, ref, devices=devices)
    monkeypatch.setattr(engine, "plan_k_chunk", lambda *a, **k: 1024)
    _check_coexnet(dt, dc, 0.05, _reference(dt, dc, 0.05), devices="all")
