"""Host-side logic that needs no GPU: covariate basis, tile lists, single=4 closed form,
digit slicing arithmetic, argument validation, the C-ABI library's symbol table."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import normalisr_oracle as orc
from conftest import ROOT, assert_p_close, load_golden
from normalisr_b200 import _lib, association, engine, single4


def test_covariate_basis_is_reference_projection():
    g = load_golden("coex_rankdef")
    dc, dt = g["dc"], g["dt"]
    Qt, rank, W = association.covariate_basis(dc)
    dci, dcr = orc.pinv_rank(dc @ dc.T)
    assert rank == dcr == 4
    np.testing.assert_allclose(Qt @ Qt.T, np.eye(rank), atol=1e-13)
    ref = dt - (dci @ (dc @ dt.T)).T @ dc          # association.py:226-229
    mine = dt - (dt @ Qt.T) @ Qt
    np.testing.assert_allclose(mine, ref, atol=1e-10)
    # W maps basis coefficients to covariate coefficients: same fitted values
    np.testing.assert_allclose((dt @ Qt.T) @ W @ dc, (dt @ Qt.T) @ Qt, atol=1e-9)


def test_covariate_basis_empty_and_zero():
    assert association.covariate_basis(np.zeros((0, 10)))[1] == 0
    assert association.covariate_basis(np.zeros((3, 10)))[1] == 0


def test_inv_rank_matches_oracle():
    rng = np.random.default_rng(3)
    c = rng.normal(size=(6, 40))
    c[5] = c[0] - c[1]
    a, ra = association.inv_rank(c @ c.T)
    b, rb = orc.pinv_rank(c @ c.T)
    assert ra == rb == 5
    np.testing.assert_allclose(a, b, atol=1e-12)
    with pytest.raises(ValueError):
        association.inv_rank(np.zeros((2, 3)))
    with pytest.raises(NotImplementedError):
        association.inv_rank(np.stack([np.eye(3)] * 2), mpc=2)               # association.py:58-60
    with pytest.raises(ValueError):
        association.inv_rank(np.eye(3), method='scipys')
    for bad in (dict(tol=0), dict(qr=-1), dict(qr=1.5)):
        with pytest.raises(ValueError):
            association.inv_rank(np.eye(3), **bad)


def test_inv_rank_every_option_matches_reference():
    """Rank cap, exact and randomised truncated SVD (random_state 0), QR-normalised power iterations, stacks
    (association.py:4-134), against tests/golden/inv_rank.npz made by the unmodified reference."""
    import json
    from conftest import load_golden
    g = load_golden("inv_rank")
    options = json.loads(str(g["options"]))
    for i in range(4):
        for j, ka in enumerate(options):
            inv, rank = association.inv_rank(g["m%d" % i], **ka)
            want = g["inv%d_%d" % (i, j)]
            assert rank == int(g["rank%d_%d" % (i, j)]), (i, ka)
            np.testing.assert_allclose(inv, want, rtol=1e-9, atol=1e-11 * np.abs(want).max(), err_msg=str((i, ka)))
    inv, rank = association.inv_rank(g["stack"])
    np.testing.assert_allclose(inv, g["stack_inv"], rtol=1e-9, atol=1e-12)
    assert np.array_equal(rank, g["stack_rank"])


def test_tile_lists_cover_exactly_once():
    for rows in (1, 128, 129, 1000, 5000):
        t = engine.coex_tiles(rows)
        nt = (rows + 127) // 128
        assert len(t) == nt * (nt + 1) // 2
        assert len({tuple(x) for x in t}) == len(t) and (t[:, 0] <= t[:, 1]).all()
    t = engine.rect_tiles(300, 1000)
    assert len(t) == 3 * 8 and len({tuple(x) for x in t}) == 24


def _upper_loop(js_range, col_end, rows_of, strip=12):
    out = []
    for js in js_range:
        je = min(js + strip, col_end)
        for i in rows_of(je):
            for j in range(max(i, js), je):
                out.append((i, j))
    return np.asarray(out, dtype=np.int32).reshape(-1, 2)


def test_upper_tiles_equal_the_three_tile_lists_it_replaces():
    """One generator stands for three tile lists whose ORDER is the L2 plan of the contraction: the full upper
    triangle (``coex_tiles``), the tiles of a column range (the streamed host pipeline) and the upper triangle of a
    strip of tile rows (the all-gather schedule's ``strip_tiles``).  Expected values are those functions' loops."""
    from normalisr_b200 import parallel
    for rows in (1, 128, 129, 1000, 1900, 5000, 12345, 20000):
        t = (rows + 127) // 128
        want = _upper_loop(range(0, t, 12), t, lambda je: range(0, je))
        assert np.array_equal(engine.coex_tiles(rows), want)
        for world in range(1, 9):
            for a, b in parallel.strip_bounds(t, world):
                want = _upper_loop(range(a, t, 12), t, lambda je: range(a, min(b, je)))
                got = parallel.strip_tiles(t, a, b)
                assert got.dtype == np.int32 and np.array_equal(got, want), (rows, world, a, b)
    for t0, t1 in ((0, 1), (0, 12), (0, 13), (3, 5), (5, 29), (12, 24), (40, 157), (150, 157), (7, 7)):
        want = _upper_loop(range(t0, t1, 12), t1, lambda je: range(0, je))
        assert np.array_equal(engine.upper_tiles(0, t1, t0, t1), want), (t0, t1)


@pytest.mark.parametrize("case", ["de_single4", "de_single4_rankdef"])
def test_single4_closed_form_equals_reference(case):
    """loo_stats on exact float64 Gram matrices reproduces the reference's single=4 numbers."""
    g = load_golden(case)
    dg, dt, dc = g["dg"], g["dt"], g["dc"]
    keep = np.array([len(np.unique(x)) > 1 for x in dg])
    dx = dg[keep]
    n = dx.shape[1]
    Qt, rank_c, _ = association.covariate_basis(dc)
    rx = dx - (dx @ Qt.T) @ Qt
    ry = dt - (dt @ Qt.T) @ Qt
    dxx, dxy, dyy, rank, w = single4.loo_stats(torch.from_numpy(rx @ rx.T), torch.from_numpy(rx @ ry.T),
                                               torch.from_numpy((ry ** 2).sum(1)), n, rank_c)
    gamma = (dxy / dxx[:, None]).numpy()
    np.testing.assert_allclose(gamma, g["gamma"][keep], rtol=1e-7, atol=1e-12)
    np.testing.assert_allclose(dxx.numpy(), g["varg"][keep], rtol=1e-9)
    np.testing.assert_allclose(dyy.numpy(), g["vart"][keep], rtol=1e-9)
    r2 = (dxy * dxy / (dxx[:, None] * dyy)).numpy()
    P = orc.beta_cdf(1 - r2, ((n - 1 - rank.numpy()) / 2)[:, None])
    assert_p_close(P, g["P"][keep], rtol=1e-6)


def test_single4_rank_deficient_groupings_fall_back():
    rng = np.random.default_rng(5)
    n = 300
    dx = (rng.random((5, n)) < 0.2).astype(float)
    dx[4] = dx[0] + dx[1]                       # exactly collinear grouping
    ry = rng.normal(size=(7, n))
    G = torch.from_numpy(dx @ dx.T)
    out = single4.loo_stats(G, torch.from_numpy(dx @ ry.T), torch.from_numpy((ry ** 2).sum(1)), n, 0)
    assert out[3].max() < 4 + 1e-9              # per-x rank is reduced, as inv_rank reports


def test_products_and_chunk_planner_arithmetic():
    assert sorted(len(v) for v in engine.products_of(3, 8).values()) == [1, 2, 2, 3]
    assert sum(len(v) for v in engine.products_of(3, 6).values()) == 6
    assert sum(len(v) for v in engine.products_of(4, 10).values()) == 10

    class Fake:                      # just the attributes plan_k_chunk reads
        n, n_pad, n_slices = 100000, 100096, 3
    ks = engine._lib.load().nsr_cell_splits(100000)
    assert ks == 49
    e = np.zeros((64, 4))
    e[:ks, 0] = 450 * 2048          # plane 0: small digits after Hadamard mixing
    e[:ks, 1:3] = 5461 * 2048       # lower planes: uniform digits
    assert engine.plan_k_chunk(Fake, Fake, 8, energies=(e, e)) == 0
    worst = np.zeros((64, 4))
    worst[:ks, :3] = 128 * 128 * 2048      # every digit +-128: 3 products * 16384 * 100096 > 2^31
    kc = engine.plan_k_chunk(Fake, Fake, 8, energies=(worst, worst))
    assert 0 < kc <= 43690 and kc % 128 == 0


def test_digit_slicing_roundtrip():
    """Balanced base-256 digits (nsr_common.cuh nsr_digits) restated in numpy."""
    rng = np.random.default_rng(0)
    for s in (2, 3, 4):
        vmax = 127 * 256 ** (s - 1)
        v = np.concatenate([rng.integers(-vmax, vmax + 1, size=5000), [vmax, -vmax, 0, 127, 128, -128, -129]])
        digits = []
        w = v.copy()
        for _ in range(s - 1):
            d = ((w + 128) % 256) - 128
            digits.append(d)
            w = (w - d) // 256
        digits.append(w)
        digits = digits[::-1]
        assert all(np.abs(d).max() <= 128 for d in digits) and np.abs(digits[0]).max() <= 127
        back = sum(d * 256 ** (s - 1 - i) for i, d in enumerate(digits))
        np.testing.assert_array_equal(back, v)


def test_argument_validation_needs_no_gpu():
    x = np.zeros((3, 10))
    with pytest.raises(ValueError):
        association.association_tests(x, None, np.ones((1, 9)))
    with pytest.raises(ValueError):
        association.association_tests(x, None, np.ones((1, 10)), single=7)
    with pytest.raises(NotImplementedError):
        association.association_tests(x, x, np.ones((1, 10)), single=5)
    with pytest.raises(NotImplementedError):
        association.association_tests(x, None, np.ones((1, 10)), single=1)
    with pytest.raises(ValueError):
        association.association_tests(x, None, np.ones((1, 10)), dimreduce=np.zeros(3))


def test_library_exports_every_declared_symbol():
    """The C-ABI library loads (no compute without a GPU) and exports what include/*.h declares."""
    header = open(os.path.join(ROOT, "include", "normalisr_b200.h")).read()
    declared = set(re.findall(r"\b(nsr_[a-z_0-9]+)\s*\(", header))
    assert declared == set(_lib.exported_symbols()), declared ^ set(_lib.exported_symbols())
    lib = _lib.load()
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.nsr_version() == 100
    assert lib.nsr_padded_cells(1) == 128 and lib.nsr_padded_cells(128) == 128 and lib.nsr_padded_cells(129) == 256


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback():
    g = load_golden("coex_nocov")
    with pytest.raises(Exception) as e:
        association.association_tests(g["dt"], None, g["dc"])
    assert "CUDA" in str(e.value) or "cuda" in str(e.value)


@pytest.mark.parametrize("case", ["de_single1", "de_single1_alpha", "de_single1_rankdef", "de_single1_nocov"])
def test_single1_sufficient_statistics_equal_reference(case):
    """The decomposition single1.py relies on (sums over S_x = sums over U + sums over T_x, closed
    form with the pseudo-inverse of the subset's covariate Gram matrix), in plain numpy, against the
    reference's per-x subset regression."""
    from scipy.special import betainc
    g = load_golden(case)
    keep = np.array([len(np.unique(x)) > 1 for x in g["dg"]])
    dx, dy, dc = g["dg"][keep], g["dt"], g["dc"]
    dimreduce = int(g["dimreduce"]) if "dimreduce" in g else 0
    nx, nc = dx.shape[0], dc.shape[0]
    colsum = dx.sum(0)
    in_u = colsum == 0
    owner = np.where(colsum == 1, dx.argmax(0), nx)
    c_u = dc[:, in_u] @ dc[:, in_u].T
    cy_u, yy_u = dy[:, in_u] @ dc[:, in_u].T, (dy[:, in_u] ** 2).sum(1)
    for x in range(nx):
        t = np.nonzero(owner == x)[0]
        ns = in_u.sum() + len(t)
        ct = dc[:, t]
        cx = ct.sum(1)
        ci, r = association.inv_rank(c_u + ct @ ct.T) if nc else (np.zeros((0, 0)), 0)
        ccx = ci @ cx
        vx = (len(t) - cx @ ccx) / ns
        cy = cy_u + dy[:, t] @ ct.T
        ccy = cy @ ci
        vy = (yy_u + (dy[:, t] ** 2).sum(1) - (ccy * cy).sum(1)) / ns
        gam = (dy[:, t].sum(1) - ccy @ cx) / (ns * vx)
        P = betainc((ns - 1 - r - dimreduce) / 2, 0.5, 1 - gam * gam * vx / vy)
        row = np.nonzero(keep)[0][x]
        np.testing.assert_allclose(P, g["P"][row], rtol=1e-9)
        np.testing.assert_allclose(gam, g["gamma"][row], rtol=1e-9, atol=1e-13)
        np.testing.assert_allclose(vx, g["varg"][row], rtol=1e-11)
        np.testing.assert_allclose(vy, g["vart"][row], rtol=1e-11)
        if "alpha" in g:
            np.testing.assert_allclose(ccy - gam[:, None] * ccx[None, :], g["alpha"][row], atol=1e-11)


def test_single1_batched_pinv_matches_inv_rank():
    from normalisr_b200 import single1
    rng = np.random.default_rng(12)
    mats = []
    for k in range(20):
        a = rng.normal(size=(6, 40))
        if k % 3 == 0:
            a[2] = a[0] - 2 * a[5]                     # rank 5
        if k % 7 == 0:
            a[4] = 0                                   # a zero covariate
        mats.append(a @ a.T)
    inv, rank = single1._pinv_rank_batched(np.array(mats))
    for m, i, r in zip(mats, inv, rank):
        want, r0 = association.inv_rank(m)
        assert r == r0
        np.testing.assert_allclose(i, want, rtol=1e-9, atol=1e-12 * np.abs(want).max())


def test_every_module_imports_without_a_gpu():
    """The package (and the reference-shaped namespace) must import on a CPU-only box: the driver's
    build check does exactly that."""
    import importlib
    for name in ("normalisr", "association", "coex", "de", "single1", "single4", "binnet", "norm", "lcpm",
                 "parallel", "engine", "synth", "_build", "_lib"):
        importlib.import_module("normalisr_b200." + name)
    import normalisr_b200.normalisr as norm
    assert set(norm.__all__) == {"coex", "de", "binnet", "normvar", "lcpm", "compute_var"}


def test_host_copy2d_thread_team():
    """nsr_host_copy2d (the staging copy between pageable arrays and page-locked slots): strided source and
    destination, short and long rows, one thread and many; a host function, no CUDA call inside."""
    import torch
    from normalisr_b200 import hoststage
    g = torch.Generator().manual_seed(5)
    for rows, cols, threads in ((1, 7, 0), (3000, 600, 0), (40, 300000, 3), (2500, 1100, 1), (0, 5, 0)):
        src_big = torch.randn((rows + 3, cols + 5), generator=g, dtype=torch.float64)
        dst_big = torch.zeros((rows + 2, cols + 9), dtype=torch.float64)
        src, dst = src_big[2:2 + rows, 1:1 + cols], dst_big[1:1 + rows, 4:4 + cols]
        hoststage.host_copy2d(dst, src, threads)
        assert torch.equal(dst, src)
        assert int((dst_big != 0).sum()) == int((src != 0).sum())           # nothing written outside the block
    a = torch.arange(12, dtype=torch.float64).reshape(3, 4)
    b = torch.empty_like(a)
    hoststage.host_copy2d(b, a)
    assert torch.equal(a, b)


def test_constant_rows_filter_and_single4_keyword_rules():
    """de.py:92-93 (len(np.unique(x)) > 1 per grouping) without full passes over the matrix; the inv_rank keywords
    single=4 accepts (those under which the reference computes the exact pseudo-inverse)."""
    from normalisr_b200 import de as de_mod, single4
    rng = np.random.default_rng(2)
    d = (rng.random((40, 9000)) < 0.01).astype(float)
    d[3] = 0
    d[5] = 1
    d[7] = 0
    d[7, -1] = 2.5                                   # differs only in the last column
    d[9] = -3.25
    want = np.array([len(np.unique(x)) > 1 for x in d])
    assert np.array_equal(de_mod._rows_that_vary(d), want)
    assert np.array_equal(de_mod._rows_that_vary(d[:, :1]), np.zeros(40, dtype=bool))
    assert de_mod._rows_that_vary(np.zeros((3, 0))).tolist() == [False] * 3
    for ka in (dict(), dict(mpc=0), dict(mpc=12, method="scipy"), dict(mpc=500, qr=3), dict(method="auto")):
        ka = dict(ka)
        single4._exact_inverse_only(ka, 12)
        assert not ka                                 # consumed
    for ka in (dict(mpc=11), dict(method="sklearn"), dict(mpc=3, method="scipy")):
        with pytest.raises(NotImplementedError):
            single4._exact_inverse_only(dict(ka), 12)
