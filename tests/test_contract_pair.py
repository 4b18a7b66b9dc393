"""The cta_group::2 pair kernel (``umma_pair``): a CTA pair computes 256 x 128 output tiles.

Integer sums do not depend on the order of the products, so the pair kernel, the single-CTA
tcgen05 kernel (``umma_pair=0``) and the CUDA-core dp4a engine must give the same P and dot bit
for bit, at every precision preset, tile count and cell chunking.
"""
import ctypes

import numpy as np
import pytest
import torch

from normalisr_b200 import _lib, association, engine, synth


def _planes(rows, n, precision, seed=1201):
    ctx = engine.context(0)
    p = synth.device_problem(seed, rows, n, "cuda")
    Qt, rank, _ = association.covariate_basis(p["dc"].cpu().numpy())
    S, prods = engine.PRESETS[precision]
    A = engine.residualize(ctx, p["dt"], torch.from_numpy(Qt).cuda(), S)
    return ctx, A, (n - 1 - rank) / 2, prods


def _run(ctx, A, dof, prods, eng, pair, k_chunk=None):
    rows = A.rows
    P = torch.zeros((rows, rows), dtype=torch.float64, device="cuda")
    D = torch.zeros_like(P)
    engine.set_option("umma_pair", pair)
    try:
        engine.contract(ctx, engine.MODE_COEX, A, A, engine.coex_tiles(rows), dof, P, D, prods, eng, k_chunk=k_chunk)
        torch.cuda.synchronize()
    finally:
        engine.set_option("umma_pair", -1)        # the default
    return P, D


# 157 tiles (odd), 1 tile, 3 tiles, 8 tiles with a partial last one
@pytest.mark.gpu
@pytest.mark.parametrize("rows,n", [(20000, 256), (100, 1000), (300, 700), (1000, 3000)])
@pytest.mark.parametrize("precision", ["default", "fast", "precise"])
def test_pair_kernel_bit_identical(rows, n, precision):
    ctx, A, dof, prods = _planes(rows, n, precision)
    Pp, Dp = _run(ctx, A, dof, prods, engine.ENGINE_UMMA, 1)
    Ps, Ds = _run(ctx, A, dof, prods, engine.ENGINE_UMMA, 0)
    assert torch.equal(Pp, Ps) and torch.equal(Dp, Ds)
    Pd, Dd = _run(ctx, A, dof, prods, engine.ENGINE_SIMT, 0)
    assert torch.equal(Pp, Pd) and torch.equal(Dp, Dd)
    assert torch.equal(Pp, Pp.T) and torch.equal(Dp, Dp.T)
    assert bool((torch.diagonal(Pp) == 0).all())


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["default", "precise"])
def test_pair_kernel_cell_chunks(precision):
    """Forced cell chunks: each chunk's integer sums and the float64 running sum between chunks are
    formed in the same order by both tcgen05 kernels."""
    ctx, A, dof, prods = _planes(1500, 5000, precision)
    for kc in (128, 1024):
        Pp, Dp = _run(ctx, A, dof, prods, engine.ENGINE_UMMA, 1, k_chunk=kc)
        Ps, Ds = _run(ctx, A, dof, prods, engine.ENGINE_UMMA, 0, k_chunk=kc)
        assert torch.equal(Pp, Ps) and torch.equal(Dp, Ds)


@pytest.mark.gpu
def test_pair_kernel_static_and_dynamic_claiming_agree():
    ctx, A, dof, prods = _planes(2500, 2048, "default")
    outs = []
    try:
        for dyn in (1, 0):
            engine.set_option("umma_dynamic", dyn)
            outs.append(_run(ctx, A, dof, prods, engine.ENGINE_UMMA, 1))
    finally:
        engine.set_option("umma_dynamic", 1)
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])



def _pair_tiles(tiles, symmetric):
    tiles = np.ascontiguousarray(tiles, dtype=np.int32)
    out = np.full((max(len(tiles), 1), 3), -7, dtype=np.int32)
    k = _lib.load().nsr_pair_tiles(tiles.ctypes.data_as(ctypes.c_void_p), len(tiles), int(symmetric),
                                   out.ctypes.data_as(ctypes.c_void_p))
    return out[:k]


def _covered(entries):
    """Unordered block pairs the entries compute (one per CTA that is not idle), and the idle CTAs."""
    got = [(min(r, c), max(r, c)) for r0, r1, c in entries for r in (r0, r1) if r >= 0]
    return got, sum(1 for e in entries if e[1] < 0)


@pytest.mark.parametrize("rows", [1, 100, 129, 300, 1000, 5000, 20000])
def test_pair_tiles_cover_every_block_pair_once(rows):
    tiles = engine.coex_tiles(rows)
    want = sorted((int(i), int(j)) for i, j in tiles)
    for sym in (0, 1):
        ent = _pair_tiles(tiles, sym)
        assert (ent[:, 0] >= 0).all() and (ent[:, 1] >= -1).all()
        got, idle = _covered(ent)
        assert sorted(got) == want                       # every block pair exactly once
        if not sym:                                      # no transposed tiles
            assert all(r <= c for r0, r1, c in ent for r in (r0, r1) if r >= 0)
    # with transposed tiles at most one CTA of one entry is idle: the columns with an odd tile count are
    # matched two by two
    t = (rows + 127) // 128
    assert idle == ((t + 1) // 2) % 2


def test_pair_tiles_of_any_subset_and_order():
    tiles = engine.coex_tiles(3000)
    rng = np.random.default_rng(3)
    for part in np.array_split(rng.permutation(len(tiles)), 5):
        sub = tiles[part]
        for sym in (0, 1):
            got, _ = _covered(_pair_tiles(sub, sym))
            assert sorted(got) == sorted((int(i), int(j)) for i, j in sub)
    assert len(_pair_tiles(tiles[:0], 1)) == 0


def test_pair_tiles_keep_the_callers_order():
    """Entries come in the order the caller's list first reaches them (the column strips' L2 plan)."""
    tiles = engine.coex_tiles(20000)
    first = {(int(i), int(j)): t for t, (i, j) in enumerate(tiles)}
    ent = _pair_tiles(tiles, 1)
    pos = [min(first[(min(r, c), max(r, c))] for r in (r0, r1) if r >= 0) for r0, r1, c in ent]
    assert pos == sorted(pos)
