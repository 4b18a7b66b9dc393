"""``coextop`` on several GPUs (``parallel.coextop_all_devices``): the strips of tile rows dealt out to the GPUs,
each GPU's partial top-k lists merged by the owner of the rows (csrc/topk_merge.cu ``nsr_topk_reset`` +
``nsr_topk_merge``).  CPU: the C ABI, the kernels' register use, and the dealing.  GPU: the merge kernel against
numpy on hand-built parts; every world size emulated on one device; the team path on one device; and, where
the box has them, several devices, each bit-identical to one-GPU ``coextop``."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT

gpu = pytest.mark.gpu
INT_MAX = 2 ** 31 - 1
SLOT = np.dtype([("key", "<f8"), ("p", "<f8"), ("dot", "<f8"), ("col", "<i4"), ("pad", "<i4")])


# --------------------------------------------------------------------------------------------------- CPU
def test_merge_entry_points_in_the_abi():
    from normalisr_b200 import _lib
    lib = _lib.load()
    for name in ("nsr_topk_reset", "nsr_topk_merge"):
        assert name in _lib.exported_symbols() and getattr(lib, name).argtypes
    header = open(os.path.join(ROOT, "include", "normalisr_b200.h")).read()
    assert "int nsr_topk_reset(" in header and "int nsr_topk_merge(" in header
    assert "#define NSR_TOPK_MAX_PARTS %d" % _lib.TOPK_MAX_PARTS in header


@pytest.mark.skipif(shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"),
                    reason="needs nvcc")
def test_merge_kernels_do_not_spill(tmp_path):
    """The reset kernel and both merge kernels (a warp per row, a CTA per row) of csrc/topk_merge.cu compile for
    sm_100a without local-memory spills or a stack frame."""
    from normalisr_b200 import _build
    res = subprocess.run([_build._nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17",
                          "-Xptxas", "-v", "-c", "-o", str(tmp_path / "topk_merge.o"),
                          os.path.join(_build.CSRC, "topk_merge.cu")], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-2000:]
    entries = re.findall(r"Compiling entry function '(\w+)'", res.stderr)
    spills = re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", res.stderr)
    frames = re.findall(r"(\d+) bytes stack frame", res.stderr)
    assert sum("topk_merge_kernel" in e for e in entries) == 2 and any("topk_reset_kernel" in e for e in entries)
    assert len(spills) >= len(entries) == 3
    assert all(s == ("0", "0") for s in spills), spills
    assert all(f == "0" for f in frames), frames


@pytest.mark.parametrize("world", range(1, 9))
def test_coextop_deal_covers_everything_once(world):
    """Every upper tile belongs to one GPU's strips, every row to one owner block; a GPU holds the planes of
    every row its strips read (its own block and its pulls), and the owner of a row merges the selection of
    every GPU whose strips reach that row.  From fewer tile rows than GPUs (empty ranges) to 1,900 genes."""
    from normalisr_b200 import parallel
    from normalisr_b200._lib import TILE
    for G in (2, 130, 300, 700, 1000, 1900):
        t = (G + TILE - 1) // TILE
        deal = parallel.coextop_deal(G, world)
        assert len(deal) == world
        owner_of_tile_row = np.full(t, -1)
        for w, d in enumerate(deal):
            assert 0 <= d.a <= d.b <= t
            assert owner_of_tile_row[d.a:d.b].tolist() == [-1] * (d.b - d.a)
            owner_of_tile_row[d.a:d.b] = w
        assert (owner_of_tile_row >= 0).all()
        owner_of_row = np.full(G, -1)
        for w, d in enumerate(deal):
            assert (owner_of_row[d.lo:d.hi] == -1).all()
            owner_of_row[d.lo:d.hi] = w
        assert (owner_of_row >= 0).all()
        for w, d in enumerate(deal):
            held = np.zeros(G, bool)
            held[d.lo:d.hi] = True
            for s in d.pulls:
                assert s != w and deal[s].hi > deal[s].lo
                held[deal[s].lo:deal[s].hi] = True
            if d.b > d.a:
                assert held[d.a * TILE:].all(), (G, world, w)
            else:
                assert d.pulls == []
        for ti in range(t):
            w = owner_of_tile_row[ti]
            for tj in range(ti, t):
                for r in (ti * TILE, min(tj * TILE, G - 1), min(ti * TILE + TILE, G) - 1, min(tj * TILE + TILE, G) - 1):
                    assert w in deal[owner_of_row[r]].parts, (G, world, ti, tj, r)
        for d in deal:
            assert len(d.parts) == len(set(d.parts)) and all(deal[w].b > deal[w].a for w in d.parts)


# --------------------------------------------------------------------------------------------------- GPU
def _slots(key, col, p, dot):
    """(rows, k, 4) float64 array of 32-byte slots from (rows, k) fields; col INT_MAX marks an empty slot."""
    s = np.zeros(key.shape, dtype=SLOT)
    s["key"], s["col"], s["p"], s["dot"] = key, col, p, dot
    return s.view(np.float64).reshape(key.shape + (4,))


def _make_parts(rng, rows, k, n_parts, short_row=None):
    """Random partial selections with ties: per row, distinct columns dealt to the parts at random; keys from a
    few values, so equal keys meet in different parts; each part keeps at most k, sorted; some parts come out
    empty or partly filled.  The row ``short_row`` gets fewer than k filled slots in all.  Returns the parts and
    the expected (idx, P_k, dot_k) of their union."""
    key = np.full((n_parts, rows, k), -1.0)
    col = np.full((n_parts, rows, k), INT_MAX, dtype=np.int64)
    p = np.zeros((n_parts, rows, k))
    dot = np.zeros((n_parts, rows, k))
    want = [np.zeros((rows, k), np.int64), np.zeros((rows, k)), np.zeros((rows, k))]
    for r in range(rows):
        n_cand = k - 1 if r == short_row else int(rng.integers(k, k * min(n_parts, 3) + 1))
        cols = rng.choice(10 * k * n_parts + 10, n_cand, replace=False)
        keys = rng.integers(0, 4, n_cand) / 4.0
        owner = rng.integers(0, n_parts, n_cand)
        if n_parts > 2:
            owner[owner == 1] = 0                 # part 1 stays empty in every row
        ps, ds = rng.standard_normal(n_cand), rng.standard_normal(n_cand)
        for q in range(n_parts):
            m = np.flatnonzero(owner == q)
            o = m[np.lexsort((cols[m], -keys[m]))][:k]
            key[q, r, :len(o)], col[q, r, :len(o)] = keys[o], cols[o]
            p[q, r, :len(o)], dot[q, r, :len(o)] = ps[o], ds[o]
        o = np.lexsort((cols, -keys))[:k]
        if r != short_row:
            want[0][r], want[1][r], want[2][r] = cols[o], ps[o], ds[o]
    parts = [_slots(key[q], col[q], p[q], dot[q]) for q in range(n_parts)]
    return parts, want


@gpu
@pytest.mark.parametrize("n_parts", [1, 2, 3, 8, 16])
@pytest.mark.parametrize("k", [1, 7, 2048])
def test_merge_kernel_against_numpy(n_parts, k):
    """The union of the parts' filled slots, best k in rank order, bit for bit; ties broken by the column."""
    from normalisr_b200 import engine
    ctx = engine.context(0)
    rng = np.random.default_rng(1000 * n_parts + k)
    rows = 3 if k == 2048 else 300
    parts, want = _make_parts(rng, rows, k, n_parts)
    got = engine.topk_merge(ctx, [torch.from_numpy(s).cuda() for s in parts])
    for g, w in zip(got, want):
        assert np.array_equal(g.cpu().numpy().view(np.int64), w.view(np.int64))


@gpu
def test_merge_kernel_short_row_raises():
    """A row whose parts hold fewer than k filled slots in all: the launch reports it and the host raises."""
    from normalisr_b200 import _lib, engine
    ctx = engine.context(0)
    for k, n_parts in ((7, 3), (300, 2)):
        parts, _ = _make_parts(np.random.default_rng(k), 40, k, n_parts, short_row=17)
        with pytest.raises(_lib.NsrError, match="fewer than k"):
            engine.topk_merge(ctx, [torch.from_numpy(s).cuda() for s in parts])


@gpu
def test_reset_sets_every_slot_empty():
    from normalisr_b200 import engine
    ctx = engine.context(0)
    state = torch.full((37, 9, 4), 5.0, dtype=torch.float64, device="cuda")
    engine.topk_reset(ctx, state)
    s = state.cpu().numpy().reshape(-1, 4).view(SLOT).ravel()
    assert (s["key"] == -1.0).all() and (s["col"] == INT_MAX).all()
    assert (s["p"] == 0).all() and (s["dot"] == 0).all() and (s["pad"] == 0).all()


KS = (1, 7, 100, 1899)


@pytest.fixture(scope="module")
def problem():
    """1,900 genes (not a multiple of the 128-row tile) x 3,000 cells with planted modules (test_coextop's)."""
    from normalisr_b200 import synth
    p = synth.device_problem(1012, 1900, 3000, "cuda")
    return p["dt"].cpu().numpy(), p["dc"].cpu().numpy()


@pytest.fixture(scope="module")
def reference(problem):
    """One-GPU coextop for every k of KS."""
    from normalisr_b200 import normalisr as norm
    dt, dc = problem
    return {k: norm.coextop(dt, dc, k) for k in KS}


def _same(got, want):
    assert len(got) == len(want) == 4
    for g, w in zip(got, want):
        g = g.cpu().numpy() if isinstance(g, torch.Tensor) else g
        assert isinstance(w, np.ndarray) and g.shape == w.shape and g.dtype == w.dtype
        assert np.array_equal(g.view(np.int64), w.view(np.int64))


def _emulated(dt, dc, k, world):
    """The schedule of ``coextop_all_devices`` for ``world`` GPUs on one device: one residualised matrix, a reset
    state per emulated GPU selected over its strips (``coex.top_strips``), and one merge per owner block of the
    partial lists of the GPUs that reach it."""
    from normalisr_b200 import engine, parallel
    from normalisr_b200.association import _residualize_any, basis_and_dof
    from normalisr_b200.coex import top_strips
    ctx = engine.context(0)
    G, n = dt.shape
    n_slices, n_products = engine.PRESETS["default"]
    Qt_dev, _, _, dof_a = basis_and_dof(ctx, dc, n, 0)
    A = _residualize_any(ctx, dt, Qt_dev, n_slices, False)
    k_chunk = engine.plan_k_chunk(A, A, n_products)
    deal = parallel.coextop_deal(G, world)
    states = []
    for d in deal:
        states.append(torch.empty((G, k, 4), dtype=torch.float64, device=ctx.device))
        engine.topk_reset(ctx, states[-1])
        top_strips(ctx, A, dof_a, n_products, k_chunk, states[-1], d.a, d.b)
    out = [np.empty((G, k), np.int64), np.empty((G, k)), np.empty((G, k))]
    for d in deal:
        if d.hi > d.lo:
            for o, t in zip(out, engine.topk_merge(ctx, [states[w][d.lo:d.hi] for w in d.parts])):
                o[d.lo:d.hi] = t.cpu().numpy()
    return tuple(out) + (A.var.cpu().numpy(),)


@gpu
@pytest.mark.parametrize("world", [2, 3, 4, 8])
@pytest.mark.parametrize("strip_tiles", [1, None])
def test_emulated_worlds_equal_one_gpu(problem, reference, monkeypatch, world, strip_tiles):
    """W GPUs' strips, resets and merges on one device, strips of one tile row and of the default height, k up to
    G - 1 (more than any owner block's rows): one-GPU coextop bit for bit."""
    from normalisr_b200 import coex as cx
    dt, dc = problem
    if strip_tiles:
        monkeypatch.setattr(cx, "_STRIP_BYTES", 16 * 128 * dt.shape[0] * strip_tiles)
    for k in KS:
        _same(_emulated(dt, dc, k, world), reference[k])


@gpu
def test_emulated_worlds_forced_cell_chunks_and_ties(problem, monkeypatch):
    """The contraction in cell chunks, and duplicated genes across block boundaries with an all-zero gene: the
    emulated worlds equal one-GPU coextop under the same input and chunking."""
    from normalisr_b200 import coex as cx, engine
    from normalisr_b200 import normalisr as norm
    dt, dc = problem
    monkeypatch.setattr(cx, "_STRIP_BYTES", 16 * 128 * dt.shape[0] * 2)
    tied = dt.copy()
    tied[10] = tied[20]
    tied[1500] = tied[20]                         # blocks 0 and 1 of 2, 0 and 6 of 8
    tied[256] = tied[255]                         # blocks 0 and 1 of 8
    tied[700] = tied[699]
    tied[5] = 0.0
    for world in (2, 3, 8):
        _same(_emulated(tied, dc, 7, world), norm.coextop(tied, dc, 7))
        _same(_emulated(tied, dc, 100, world), norm.coextop(tied, dc, 100))
    monkeypatch.setattr(engine, "plan_k_chunk", lambda *a, **k: 1024)
    for world in (3, 4):
        _same(_emulated(dt, dc, 100, world), norm.coextop(dt, dc, 100))


@gpu
@pytest.mark.parametrize("chunked", [False, True])
def test_team_path_on_one_gpu(problem, reference, monkeypatch, chunked):
    """``coextop_all_devices`` on ONE device: the worker thread, the projection into the full G-row planes, the
    reset, a one-part merge and the host assembly; and ``coextop(..., devices=[0])``."""
    from normalisr_b200 import engine, parallel
    from normalisr_b200 import normalisr as norm
    dt, dc = problem
    if chunked:
        monkeypatch.setattr(engine, "plan_k_chunk", lambda *a, **k: 1024)
        ref = {k: norm.coextop(dt, dc, k) for k in (7, 100)}
    else:
        ref = reference
    for k in ((7, 100) if chunked else KS):
        _same(parallel.coextop_all_devices(dt, dc, k, devices=[0]), ref[k])
    _same(norm.coextop(dt, dc, 7, devices=[0]), ref[7])
    _same(norm.coextop(dt, dc, 7, devices=["cuda:0"]), ref[7])


@gpu
def test_devices_errors(problem):
    """Several devices take host input only, and not together with ``device``; k is checked as before."""
    from normalisr_b200 import normalisr as norm
    dt, dc = problem
    with pytest.raises(ValueError, match="host inputs"):
        norm.coextop(torch.from_numpy(dt).cuda(), torch.from_numpy(dc).cuda(), 5, devices=[0, 1])
    with pytest.raises(ValueError, match="host inputs"):
        norm.coextop(dt, dc, 5, device=0, devices=[0, 1])
    for k in (0, dt.shape[0], 2.5):
        with pytest.raises(ValueError):
            norm.coextop(dt, dc, k, devices=[0, 1])


@gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs in one process")
def test_several_devices_equal_one_gpu(problem, reference, monkeypatch):
    """Every GPU of the box, two in reverse order, three where there are three, and cell chunks forced: one-GPU
    coextop bit for bit."""
    from normalisr_b200 import engine
    from normalisr_b200 import normalisr as norm
    dt, dc = problem
    lists = ["all", [1, 0]] + ([[0, 1, 2]] if torch.cuda.device_count() >= 3 else [])
    for devices in lists:
        for k in KS:
            _same(norm.coextop(dt, dc, k, devices=devices), reference[k])
    monkeypatch.setattr(engine, "plan_k_chunk", lambda *a, **k: 1024)
    _same(norm.coextop(dt, dc, 100, devices="all"), norm.coextop(dt, dc, 100))
