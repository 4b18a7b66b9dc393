"""Every gene's k strongest co-expression partners (``coextop``; csrc/topk.cu ``nsr_topk_strip`` +
``nsr_topk_finish``).  CPU: the C ABI, the kernels' register use, and the numpy reference on hand-made ties.
GPU: ``coextop`` equal to the reference's selection on ``coex``'s P, dot and var bit for bit, for every strip
height, with the contraction in cell chunks, with tied and all-zero keys; device memory bounded by one strip;
argument errors."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT

gpu = pytest.mark.gpu


def topk_ref(P, D, var, k):
    """(idx, P_k, dot_k): per row, the k columns j != i with the largest r2 = dot^2 / (var_i var_j), key
    descending then column ascending."""
    G = D.shape[0]
    r2 = D * D / (var[:, None] * var[None, :])
    cols = np.arange(G)
    idx = np.empty((G, k), dtype=np.int64)
    for i in range(G):
        c = np.delete(cols, i)
        key = np.delete(r2[i], i)
        idx[i] = c[np.lexsort((c, -key))[:k]]
    rows = np.arange(G)[:, None]
    return idx, P[rows, idx], D[rows, idx]


# --------------------------------------------------------------------------------------------------- CPU
def test_topk_ref_on_hand_made_ties():
    """Equal keys (equal dot and var, dot of opposite signs, -0.0 against +0.0) go to the smaller column; the
    diagonal never appears."""
    var = np.array([1.0, 2.0, 2.0, 1.0, 4.0, 1.0])
    D = np.array([[9.0, 1.0, -1.0, 0.5, 2.0, -0.0],
                  [1.0, 9.0, 2.0, -0.0, 0.0, 1.0],
                  [-1.0, 2.0, 9.0, 0.0, -2.0, 1.0],
                  [0.5, -0.0, 0.0, 9.0, 1.0, -0.5],
                  [2.0, 0.0, -2.0, 1.0, 9.0, 2.0],
                  [-0.0, 1.0, 1.0, -0.5, 2.0, 9.0]])
    P = np.arange(36.0).reshape(6, 6)
    idx, P_k, D_k = topk_ref(P, D, var, 5)
    want = [[4, 1, 2, 3, 5],       # keys 1, .5, .5, .25, 0
            [2, 0, 5, 3, 4],       # 1, .5, .5, 0, 0 (-0.0 and +0.0 dot tie)
            [1, 0, 4, 5, 3],       # 1, .5, .5, .5, 0
            [0, 4, 5, 1, 2],       # .25, .25, .25, 0, 0
            [0, 5, 2, 3, 1],       # 1, 1, .5, .25, 0
            [4, 1, 2, 3, 0]]       # 1, .5, .5, .25, 0
    assert idx.tolist() == want
    assert np.array_equal(P_k, P[np.arange(6)[:, None], idx]) and np.array_equal(D_k, D[np.arange(6)[:, None], idx])
    assert all(i not in idx[i] for i in range(6))
    assert np.array_equal(topk_ref(P, D, var, 1)[0][:, 0], idx[:, 0])


def test_topk_entry_points_in_the_abi():
    from normalisr_b200 import _lib
    lib = _lib.load()
    for name in ("nsr_topk_strip", "nsr_topk_finish"):
        assert name in _lib.exported_symbols() and getattr(lib, name).argtypes
    header = open(os.path.join(ROOT, "include", "normalisr_b200.h")).read()
    assert "int nsr_topk_strip(" in header and "int nsr_topk_finish(" in header
    assert "#define NSR_TOPK_MAX %d" % _lib.TOPK_MAX in header


@pytest.mark.skipif(shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"),
                    reason="needs nvcc")
def test_topk_kernels_do_not_spill(tmp_path):
    """Both kernels of csrc/topk.cu compile for sm_100a without local-memory spills."""
    from normalisr_b200 import _build
    res = subprocess.run([_build._nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17",
                          "-Xptxas", "-v", "-c", "-o", str(tmp_path / "topk.o"),
                          os.path.join(_build.CSRC, "topk.cu")], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-2000:]
    entries = re.findall(r"Compiling entry function '(\w+)'", res.stderr)
    spills = re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", res.stderr)
    assert any("topk_strip_kernel" in e for e in entries) and any("topk_finish_kernel" in e for e in entries)
    assert len(spills) >= len(entries) == 2
    assert all(s == ("0", "0") for s in spills), spills


# --------------------------------------------------------------------------------------------------- GPU
KS = (1, 7, 100, 1899)


@pytest.fixture(scope="module")
def problem():
    """1,900 genes (not a multiple of the 128-row tile) x 3,000 cells with planted modules, and coex on it."""
    from normalisr_b200 import normalisr as norm, synth
    p = synth.device_problem(1012, 1900, 3000, "cuda")
    dt, dc = p["dt"].cpu().numpy(), p["dc"].cpu().numpy()
    return dt, dc, norm.coex(dt, dc)


def _check(dt, dc, coex_out, ks=KS, device_input=True):
    from normalisr_b200 import normalisr as norm
    P, D, var = coex_out
    inputs = [(dt, dc)]
    if device_input:
        inputs.append((torch.from_numpy(dt).cuda(), torch.from_numpy(dc).cuda()))
    for k in ks:
        want = topk_ref(P, D, var, k)
        for x, c in inputs:
            got = norm.coextop(x, c, k)
            if isinstance(x, torch.Tensor):
                assert all(t.is_cuda for t in got)
                got = tuple(t.cpu().numpy() for t in got)
            else:
                assert all(isinstance(t, np.ndarray) for t in got)
            idx, P_k, D_k, v = got
            assert idx.dtype == np.int64 and idx.shape == (dt.shape[0], k)
            assert P_k.dtype == np.float64 and D_k.dtype == np.float64
            assert np.array_equal(idx, want[0]), (k, np.argwhere(idx != want[0])[:5])
            assert np.array_equal(P_k.view(np.int64), want[1].view(np.int64)), k
            assert np.array_equal(D_k.view(np.int64), want[2].view(np.int64)), k
            assert np.array_equal(v.view(np.int64), var.view(np.int64))


@gpu
@pytest.mark.parametrize("strip_tiles", [1, 3, None])
def test_coextop_equals_selection_on_coex(problem, monkeypatch, strip_tiles):
    """numpy and CUDA input, k = 1, 7, 100, G - 1, with strips of 1 and 3 tile rows (15 and 5 strips) and the
    default (one strip): the reference's selection on coex's P, dot and var, bit for bit."""
    from normalisr_b200 import coex as cx
    dt, dc, ref = problem
    if strip_tiles:
        monkeypatch.setattr(cx, "_STRIP_BYTES", 16 * 128 * dt.shape[0] * strip_tiles)
    _check(dt, dc, ref)


@gpu
def test_coextop_forced_cell_chunks(problem, monkeypatch):
    """The contraction in cell chunks: the same selection as on coex under the same chunking."""
    from normalisr_b200 import coex as cx, engine
    from normalisr_b200 import normalisr as norm
    dt, dc, _ = problem
    monkeypatch.setattr(engine, "plan_k_chunk", lambda *a, **k: 1024)
    monkeypatch.setattr(cx, "_STRIP_BYTES", 16 * 128 * dt.shape[0] * 3)
    _check(dt, dc, norm.coex(dt, dc), ks=(7, 100), device_input=False)


@gpu
def test_coextop_ties(problem, monkeypatch):
    """Duplicated genes (equal keys in every other row) and an all-zero gene (var -> 1, dot 0: every key of
    its row is 0, so its partners come out as the first columns, ascending)."""
    from normalisr_b200 import coex as cx
    from normalisr_b200 import normalisr as norm
    dt, dc, _ = problem
    dt = dt.copy()
    dt[10] = dt[20]
    dt[1500] = dt[20]
    dt[700] = dt[699]
    dt[5] = 0.0
    ref = norm.coex(dt, dc)
    assert not ref[1][5].any() and ref[2][5] == 1.0
    monkeypatch.setattr(cx, "_STRIP_BYTES", 16 * 128 * dt.shape[0] * 3)
    _check(dt, dc, ref, ks=(7, 100))
    idx = norm.coextop(dt, dc, 100)[0]
    assert np.array_equal(idx[5], np.delete(np.arange(101), 5))


@gpu
def test_coextop_memory_is_bounded_by_one_strip(monkeypatch):
    """6,000 genes x 2,000 cells with a strip of one tile row: the device memory that coextop allocates stays
    below planes + strip + slots + 64 MB, far under the 576 MB that P and dot would take."""
    from normalisr_b200 import coex as cx, engine, synth
    from normalisr_b200 import normalisr as norm
    G, n, k = 6000, 2000, 50
    p = synth.device_problem(77, G, n, "cuda")
    dt, dc = p["dt"], p["dc"]
    monkeypatch.setattr(cx, "_STRIP_BYTES", 16 * 128 * G)
    norm.coextop(dt[:300], dc, 5)                      # contexts and the covariate basis outside the window
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    idx, P_k, D_k, var = norm.coextop(dt, dc, k)
    torch.cuda.synchronize()
    used = torch.cuda.max_memory_allocated() - base
    planes = 3 * G * engine.padded_cells(n)
    strip = 16 * 128 * G
    slots = 32 * G * k
    assert used < planes + strip + slots + (64 << 20), (used, planes, strip, slots)
    assert used < 16 * G * G
    assert idx.shape == (G, k) and bool((idx != torch.arange(G, device=idx.device)[:, None]).all())


@gpu
def test_coextop_errors(problem):
    from normalisr_b200 import normalisr as norm
    dt, dc, _ = problem
    G = dt.shape[0]
    for x, c in ((dt, dc), (torch.from_numpy(dt).cuda(), torch.from_numpy(dc).cuda())):
        for k in (0, -1, G, G + 5, 2.5):
            with pytest.raises(ValueError):
                norm.coextop(x, c, k)
        with pytest.raises(ValueError):
            norm.coextop(x[:1], c, 1)
        with pytest.raises(ValueError):
            norm.coextop(x[:, :-1], c, 5)
        with pytest.raises(ValueError):
            norm.coextop(x[0], c, 5)
        with pytest.raises(ValueError):
            norm.coextop(x, c, 5, precision="nope")
    wide = np.random.default_rng(3).random((2100, 200))
    with pytest.raises(ValueError):
        norm.coextop(wide, np.ones((1, 200)), 2049)
    assert norm.coextop(wide, np.ones((1, 200)), 2048)[0].shape == (2100, 2048)
