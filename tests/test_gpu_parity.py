"""Parity of the CUDA path with the reference, through the public API / C ABI.

Tolerances are the ones BASELINE.json states: |delta r| <= 1e-6 and relative error in P
<= 1e-4 wherever P >= 1e-300 (r = dot / sqrt(var_i var_j), coex.py:34).  Three kinds of checks:
  * against the committed golden vectors produced by the unmodified reference;
  * against the CPU oracle on seeded synthetic inputs sized so the oracle takes seconds;
  * size-independent properties at the BASELINE sizes (bit-identical integer sums between the
    tcgen05 and the CUDA-core engines, symmetry, tile-subset invariance, linearity).
"""
import numpy as np
import pytest
import torch

import normalisr_oracle as orc
import nsr_testlib as tl
from conftest import R_ATOL, assert_p_close, load_golden, pearson_from

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from normalisr_b200 import association, engine, synth
    from normalisr_b200 import normalisr as norm


def _check_coex(got, ref, p_rtol=1e-4):
    P, dot, var = got
    Pr, dotr, varr = ref
    np.testing.assert_allclose(var, varr, rtol=1e-10)
    r = pearson_from(dot, var, var)
    rr = pearson_from(dotr, varr, varr)
    assert np.abs(r - rr).max() <= R_ATOL, np.abs(r - rr).max()
    assert_p_close(P, Pr, rtol=p_rtol)
    assert (np.diag(P) == 0).all() and (np.diag(dot) == 0).all()
    assert np.array_equal(P, P.T) and np.array_equal(dot, dot.T)


def test_coex_golden_fast_preset():
    """precision='fast' drops two more digit products (6 of 9): an opt-in trade of accuracy for
    ~12 % speed with its own, looser, bounds (|dr| <= 3e-6, rel dP <= 1e-3 for n >= 400)."""
    for case in ("coex_chain", "coex_tail"):
        g = load_golden(case)
        P, dot, var = norm.coex(g["dt"], g["dc"], precision="fast")
        r = pearson_from(dot, var, var)
        assert np.abs(r - pearson_from(g["dot"], g["var"], g["var"])).max() <= 3e-6
        assert_p_close(P, g["P"], rtol=1e-3)


@pytest.mark.parametrize("precision", ["default", "precise"])
@pytest.mark.parametrize("case", ["coex_chain", "coex_tail", "coex_rankdef", "coex_nocov"])
def test_coex_golden(case, precision):
    g = load_golden(case)
    ka = {"dimreduce": int(g["dimreduce"])} if "dimreduce" in g else {}
    got = norm.coex(g["dt"], g["dc"], precision=precision, **ka)
    assert all(isinstance(x, np.ndarray) and x.dtype == np.float64 for x in got)
    _check_coex(got, (g["P"], g["dot"], g["var"]))


def test_coex_golden_simt_engine():
    g = load_golden("coex_tail")
    got = norm.coex(g["dt"], g["dc"], engine=engine.ENGINE_SIMT)
    _check_coex(got, (g["P"], g["dot"], g["var"]))


@pytest.mark.parametrize("case,ka", [("de_single0", {}), ("de_single0_alpha", {"lowmem": False}),
                                     ("de_single4", {"single": 4}), ("de_single4_rankdef", {"single": 4}),
                                     ("de_single1", {"single": 1}),
                                     ("de_single1_alpha", {"single": 1, "lowmem": False, "dimreduce": 1}),
                                     ("de_single1_rankdef", {"single": 1}), ("de_single1_nocov", {"single": 1})])
def test_de_golden(case, ka):
    g = load_golden(case)
    P, gamma, alpha, varg, vart = norm.de(g["dg"], g["dt"], g["dc"], **ka)
    np.testing.assert_allclose(varg, g["varg"], rtol=1e-7)
    np.testing.assert_allclose(vart, g["vart"], rtol=1e-7)
    # gamma = r * sqrt(vart / varg): |delta r| <= 1e-6 translates to this absolute bound
    scale = np.sqrt(g["vart"] / np.where(g["varg"] > 0, g["varg"], 1)[:, None])
    assert (np.abs(gamma - g["gamma"]) <= R_ATOL * scale + 1e-12).all()
    assert_p_close(P, g["P"])
    if "alpha" in g:
        np.testing.assert_allclose(alpha, g["alpha"], rtol=1e-5, atol=1e-5 * np.abs(g["alpha"]).max())
    else:
        assert alpha is None
    assert (P[5] == 1).all() and (gamma[5] == 0).all() and varg[5] == 0 and (vart[5] == 0).all()


def test_coex_config1_against_oracle():
    """BASELINE configs[0] shape: 2,000 cells x 1,000 genes."""
    p = synth.host_problem(1001, 1000, 2000)
    ref = orc.coex(p["dt"], p["dc"])
    got = norm.coex(p["dt"], p["dc"])
    _check_coex(got, ref)
    iu = np.triu_indices(1000, 1)
    assert (ref[0][iu] < 1e-20).sum() > 100         # the tail is exercised


def test_coex_lowmem_false_and_gamma():
    g = load_golden("coex_chain")
    ref = orc.association_tests(g["dt"], None, g["dc"], lowmem=False, return_dot=False)
    got = association.association_tests(g["dt"], None, g["dc"], lowmem=False, return_dot=False)
    np.testing.assert_allclose(got[1], ref[1], atol=1e-6 * np.abs(ref[1]).max())
    np.testing.assert_allclose(got[2], ref[2], atol=1e-6 * np.abs(ref[2]).max())
    assert got[3] is None
    assert_p_close(got[0], ref[0])


def test_de_config_like_against_oracle():
    p = synth.host_problem(1003, 600, 3000, n_group=40, group_p=0.03)
    for single in (0, 4):
        ref = orc.de(p["dg"], p["dt"], p["dc"], single=single)
        got = norm.de(p["dg"], p["dt"], p["dc"], single=single)
        assert_p_close(got[0], ref[0])
        np.testing.assert_allclose(got[3], ref[3], rtol=1e-7)
        np.testing.assert_allclose(got[4], ref[4], rtol=1e-7)
        scale = np.sqrt(ref[4] / ref[3][:, None])
        assert (np.abs(got[1] - ref[1]) <= R_ATOL * scale + 1e-12).all()


def test_de_single1_low_moi_against_oracle(monkeypatch):
    """Low-MOI screen (single=1): 40 gRNAs, 12,000 cells, 700 genes; also with genes processed in
    several chunks and with device tensors."""
    from normalisr_b200 import single1
    rng = np.random.default_rng(77)
    n, g, k = 12000, 700, 40
    dc = np.concatenate([rng.normal(size=(4, n)), (rng.random((2, n)) < 0.3).astype(float), np.ones((1, n))])
    dg = np.zeros((k, n))
    u = rng.random(n)
    has = u > 0.5
    dg[rng.integers(0, k, size=n)[has], np.nonzero(has)[0]] = 1
    two = np.nonzero(u > 0.93)[0]
    dg[rng.integers(0, k, size=two.size), two] = 1
    dt = rng.normal(size=(g, n)) + 0.3 * dc[1] + 4.0
    dt[:k] += np.linspace(0, 2.5, k)[:, None] * dg                    # P from ~1 down to < 1e-100
    ref = orc.de(dg, dt, dc, single=1, lowmem=False)
    for chunk in (1 << 29, 8 * k * 9 * 100):
        monkeypatch.setattr(single1, "_CHUNK_BYTES", chunk)
        got = norm.de(dg, dt, dc, single=1, lowmem=False)
        assert_p_close(got[0], ref[0])
        np.testing.assert_allclose(got[3], ref[3], rtol=1e-9)
        np.testing.assert_allclose(got[4], ref[4], rtol=1e-9)
        scale = np.sqrt(ref[4] / ref[3][:, None])
        assert (np.abs(got[1] - ref[1]) <= R_ATOL * scale + 1e-12).all()
        np.testing.assert_allclose(got[2], ref[2], atol=1e-8 * np.abs(ref[2]).max())
    assert ref[0].min() < 1e-100
    dev = norm.de(torch.from_numpy(dg).cuda(), torch.from_numpy(dt).cuda(), torch.from_numpy(dc).cuda(), single=1)
    assert dev[0].is_cuda and dev[2] is None
    assert_p_close(dev[0].cpu().numpy(), ref[0])
    # more than 16 covariates: the closed form runs as batched tensor operations instead of the fused kernel
    dc20 = np.concatenate([dc, rng.normal(size=(13, n))])
    ref20 = orc.de(dg[:8], dt[:60], dc20, single=1, lowmem=False)
    got20 = norm.de(dg[:8], dt[:60], dc20, single=1, lowmem=False)
    assert_p_close(got20[0], ref20[0])
    np.testing.assert_allclose(got20[4], ref20[4], rtol=1e-9)
    np.testing.assert_allclose(got20[2], ref20[2], atol=1e-8 * np.abs(ref20[2]).max())


def test_de_million_cells_uses_cell_chunks():
    """Config-5 cell count (1M): the int32 bound forces the contraction into cell chunks; the
    result still matches the float64 oracle."""
    rng = np.random.default_rng(31)
    n, g, k = 1_000_000, 24, 6
    dc = np.concatenate([rng.normal(size=(2, n)), np.ones((1, n))])
    dg = (rng.random((k, n)) < 0.002).astype(np.float64)
    dt = rng.normal(size=(g, n)) + 2.0
    dt[:k] += 0.05 * dg                                    # effects: P spans ~1 .. 1e-50
    ref = orc.de(dg, dt, dc)
    got = norm.de(dg, dt, dc)
    assert_p_close(got[0], ref[0])
    np.testing.assert_allclose(got[3], ref[3], rtol=1e-7)
    np.testing.assert_allclose(got[4], ref[4], rtol=1e-7)
    scale = np.sqrt(ref[4] / ref[3][:, None])
    assert (np.abs(got[1] - ref[1]) <= R_ATOL * scale + 1e-12).all()
    # and the planner did ask for chunks at this size
    ctx = engine.context(0)
    Qt, rank, _ = association.covariate_basis(dc)
    A = engine.residualize(ctx, torch.from_numpy(dt).cuda(), torch.from_numpy(Qt).cuda(), 3)
    assert engine.plan_k_chunk(A, A, 8) > 0


def test_host_pipeline_many_chunks_equals_device_path(monkeypatch):
    """The end-to-end path for host matrices (row chunks staged on a copy stream, tiles contracted
    as their columns arrive, finished blocks copied back on a third stream, geometric tail chunks)
    gives the same bits as the device-resident path, with and without caller-provided pinned
    output buffers."""
    monkeypatch.setattr(association, "_PIPE_CHUNK_BYTES", 1)               # smallest row chunks: 256 rows each
    p = synth.host_problem(1007, 5003, 1200)
    dt_d, dc_d = torch.from_numpy(p["dt"]).cuda(), torch.from_numpy(p["dc"]).cuda()
    Pd, Dd, vd = norm.coex(dt_d, dc_d)
    Pd, Dd, vd = Pd.cpu().numpy(), Dd.cpu().numpy(), vd.cpu().numpy()
    Ph, Dh, vh = norm.coex(p["dt"], p["dc"])
    assert np.array_equal(Ph, Pd) and np.array_equal(Dh, Dd) and np.array_equal(vh, vd)
    g = p["dt"].shape[0]
    P_pin = torch.full((g, g), -1.0, dtype=torch.float64).pin_memory()
    D_pin = torch.full((g, g), -1.0, dtype=torch.float64).pin_memory()
    Po, Do, vo = norm.coex(p["dt"], p["dc"], out=(P_pin, D_pin))
    assert np.array_equal(P_pin.numpy(), Pd) and np.array_equal(D_pin.numpy(), Dd) and np.array_equal(vo, vd)
    assert np.array_equal(Po, Pd) and np.array_equal(Do, Dd)


@pytest.mark.parametrize("single", [0, 4])
def test_de_host_genes_streamed_in_row_chunks_equal_device_path(monkeypatch, single):
    """de() with a HOST expression matrix larger than one staging buffer (config 5 on one GPU: the 160 GB matrix
    never sits in HBM, only its digit planes do): the genes arrive in row chunks on a copy stream while the
    previous chunk is projected; same bits as the device-resident call."""
    p = synth.host_problem(1021, 3001, 2000, n_group=10, group_p=0.1)
    dev = norm.de(*[torch.from_numpy(p[k]).cuda() for k in ("dg", "dt", "dc")], single=single)
    monkeypatch.setattr(association, "_ROW_CHUNK_BYTES", 8 * 2000 * 257)     # 12 chunks of 257 genes
    host = norm.de(p["dg"], p["dt"], p["dc"], single=single)
    for a, b in zip(host, dev):
        if a is not None:
            assert np.array_equal(a, b.cpu().numpy())
    pinned = norm.de(p["dg"], torch.from_numpy(p["dt"]).pin_memory(), p["dc"], single=single)
    assert all(np.array_equal(a, b) for a, b in zip(pinned, host) if a is not None)


def test_host_inputs_of_any_layout_and_pinning():
    """Host matrices as the caller happens to hold them - C-ordered numpy (pageable: staged through page-locked slots
    by the thread team), Fortran-ordered numpy, a transposed CPU tensor view, page-locked tensors - give the same bits."""
    p = synth.host_problem(1023, 700, 900, n_group=8, group_p=0.1)
    want = norm.coex(p["dt"], p["dc"])
    variants = [np.asfortranarray(p["dt"]), torch.from_numpy(np.ascontiguousarray(p["dt"].T)).T,
                torch.from_numpy(p["dt"]).pin_memory()]
    for dt in variants:
        got = norm.coex(dt, p["dc"])
        assert all(np.array_equal(a, b) for a, b in zip(got, want))
    want = norm.de(p["dg"], p["dt"], p["dc"], single=4)
    for dt in variants:
        got = norm.de(np.asfortranarray(p["dg"]), dt, p["dc"], single=4)
        assert all(np.array_equal(a, b) for a, b in zip(got, want) if a is not None)


def test_device_tensors_in_device_tensors_out():
    g = load_golden("coex_chain")
    dt = torch.from_numpy(g["dt"]).cuda()
    dc = torch.from_numpy(g["dc"]).cuda()
    P, dot, var = norm.coex(dt, dc)
    assert P.is_cuda and dot.is_cuda and var.is_cuda
    _check_coex((P.cpu().numpy(), dot.cpu().numpy(), var.cpu().numpy()), (g["P"], g["dot"], g["var"]))


def test_edge_shapes():
    rng = np.random.default_rng(11)
    for (gnum, n) in [(1, 50), (2, 129), (127, 128), (129, 257), (300, 1000)]:
        dt = rng.normal(size=(gnum, n))
        dc = np.concatenate([rng.normal(size=(2, n)), np.ones((1, n))])
        _check_coex(norm.coex(dt, dc), orc.coex(dt, dc))


def test_outlier_and_degenerate_rows():
    """Rows that defeat the rms-based scale estimate: one giant spike, an all-zero row, a row that
    is an exact linear combination of covariates (residual = rounding noise in the reference,
    so only its var is compared loosely) and a very sparse gene."""
    rng = np.random.default_rng(21)
    n, g = 3000, 40
    dc = np.concatenate([rng.normal(size=(3, n)), np.ones((1, n))])
    dt = rng.normal(size=(g, n)) + 3.0
    dt[3, 777] += 5e4                       # spike: max|z'| >> 6 rms -> re-quantisation pass
    dt[5] = 0.0                             # exact zero residual: var 0 -> 1, P = 1
    dt[9] = (rng.random(n) < 0.002) * 7.0   # expressed in ~6 cells
    ref = orc.coex(dt, dc)
    got = norm.coex(dt, dc)
    _check_coex(got, ref)
    assert got[2][5] == 1.0 and (np.delete(got[0][5], 5) == 1.0).all()


def test_many_covariates():
    """rank 20 > 16: the coefficient pass needs two launches."""
    rng = np.random.default_rng(22)
    n, g = 1500, 50
    dc = np.concatenate([rng.normal(size=(19, n)), np.ones((1, n))])
    dt = rng.normal(size=(g, n)) + 0.3 * dc[:5].sum(0)
    _check_coex(norm.coex(dt, dc), orc.coex(dt, dc))


def test_more_covariates_than_the_kernels_stage():
    """rank 70 > NSR_MAX_RANK = 64: the projection falls back to float64 library GEMMs into a temporary and
    the kernels quantise without covariates - same results (coex and de, alpha included)."""
    rng = np.random.default_rng(23)
    n, g = 1200, 40
    dc = np.concatenate([rng.normal(size=(69, n)), np.ones((1, n))])
    dt = rng.normal(size=(g, n)) + 0.3 * dc[:5].sum(0)
    _check_coex(norm.coex(dt, dc), orc.coex(dt, dc))
    dg = (rng.random((6, n)) < 0.2).astype(float)
    got, want = norm.de(dg, dt, dc, lowmem=False), orc.de(dg, dt, dc, lowmem=False)
    assert_p_close(got[0], want[0])
    scale = np.sqrt(want[4] / want[3][:, None])           # gamma = r sqrt(vart / varg): the |delta r| <= 1e-6 bound
    assert (np.abs(got[1] - want[1]) <= R_ATOL * scale + 1e-12).all()
    np.testing.assert_allclose(got[2], want[2], rtol=1e-5, atol=1e-5 * np.abs(want[2]).max())


def test_errors_match_reference():
    x = np.random.default_rng(0).normal(size=(4, 5))
    with pytest.raises(ValueError):
        norm.coex(x, np.random.default_rng(1).normal(size=(4, 5)))     # n <= rank + 1
    with pytest.raises(ValueError):
        norm.coex(x, np.ones((1, 6)))
    with pytest.raises(TypeError):
        norm.coex(x, np.ones((1, 5)), nonsense=1)


# ---- properties at BASELINE sizes -------------------------------------------------------
def _sliced(rows, n, precision="default", seed=1002):
    ctx = engine.context(0)
    p = synth.device_problem(seed, rows, n, "cuda")
    Qt, rank, _ = association.covariate_basis(p["dc"].cpu().numpy())
    S, prods = engine.PRESETS[precision]
    A = engine.residualize(ctx, p["dt"], torch.from_numpy(Qt).cuda(), S)
    return ctx, p, A, rank, prods


@pytest.mark.parametrize("precision", ["default", "fast", "precise"])
def test_config2_engines_bit_identical(precision):
    """10k cells x 5k genes (BASELINE configs[1]): the tensor-core kernel must reproduce the
    CUDA-core kernel's integer sums exactly, hence identical P and dot bit patterns."""
    rows, n = 5000, 10000
    ctx, p, A, rank, prods = _sliced(rows, n, precision)
    tiles = engine.coex_tiles(rows)
    outs = []
    for eng in (engine.ENGINE_UMMA, engine.ENGINE_SIMT):
        P = torch.zeros((rows, rows), dtype=torch.float64, device="cuda")
        D = torch.zeros((rows, rows), dtype=torch.float64, device="cuda")
        engine.contract(ctx, engine.MODE_COEX, A, A, tiles, (n - 1 - rank) / 2, P, D, prods, eng)
        outs.append((P, D))
    torch.cuda.synchronize()
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    P, D = outs[0]
    assert torch.equal(P, P.T) and torch.equal(D, D.T)
    assert bool((torch.diagonal(P) == 0).all()) and bool(((P >= 0) & (P <= 1)).all())
    # a checksum of a random sample of entries against float64 inner products of the residuals
    idx = torch.randint(0, rows, (200, 2), device="cuda")
    z = p["dt"] - (p["dt"] @ torch.from_numpy(association.covariate_basis(p["dc"].cpu().numpy())[0]).cuda().T) @ \
        torch.from_numpy(association.covariate_basis(p["dc"].cpu().numpy())[0]).cuda()
    want = (z[idx[:, 0]] * z[idx[:, 1]]).sum(1) / n
    want = torch.where(idx[:, 0] == idx[:, 1], torch.zeros_like(want), want)
    got = D[idx[:, 0], idx[:, 1]]
    r_err = (got - want).abs() / torch.sqrt(A.var[idx[:, 0]] * A.var[idx[:, 1]])
    assert float(r_err.max()) < 1e-7


def test_tile_subset_invariance_and_rect_vs_sym():
    rows, n = 1500, 4096
    ctx, p, A, rank, prods = _sliced(rows, n)
    dof = (n - 1 - rank) / 2
    tiles = engine.coex_tiles(rows)
    full_P = torch.zeros((rows, rows), dtype=torch.float64, device="cuda")
    full_D = torch.zeros_like(full_P)
    engine.contract(ctx, engine.MODE_COEX, A, A, tiles, dof, full_P, full_D, prods)
    part_P = torch.zeros_like(full_P)
    part_D = torch.zeros_like(full_P)
    perm = np.random.default_rng(0).permutation(len(tiles))
    for chunk in np.array_split(perm, 3):                       # any partition, any order
        engine.contract(ctx, engine.MODE_COEX, A, A, tiles[chunk], dof, part_P, part_D, prods)
    torch.cuda.synchronize()
    assert torch.equal(full_P, part_P) and torch.equal(full_D, part_D)
    # rectangular (DE) mode on the same planes: gamma * var_x == dot off the diagonal
    gP = torch.zeros_like(full_P)
    gG = torch.zeros_like(full_P)
    engine.contract(ctx, engine.MODE_DE, A, A, engine.rect_tiles(rows, rows), dof, gP, gG, prods)
    torch.cuda.synchronize()
    off = ~torch.eye(rows, dtype=torch.bool, device="cuda")
    assert torch.equal(gP[off], full_P[off])
    torch.testing.assert_close((gG * A.var[:, None])[off], full_D[off], rtol=1e-14, atol=0)


@pytest.mark.parametrize("eng", ["umma", "simt"])
def test_cell_chunking_is_exact(eng):
    """Contracting the cells in chunks (float64 running sum between chunks) reproduces the
    single-pass result to float64 rounding, in every mode."""
    rows, n = 700, 5000
    ctx, p, A, rank, prods = _sliced(rows, n)
    e = engine.ENGINE_UMMA if eng == "umma" else engine.ENGINE_SIMT
    dof = (n - 1 - rank) / 2
    for mode, tiles in ((engine.MODE_COEX, engine.coex_tiles(rows)), (engine.MODE_DE, engine.rect_tiles(rows, rows)),
                        (engine.MODE_RAW, engine.rect_tiles(rows, rows))):
        outs = []
        for kc in (0, 128, 1024, 4096):
            P = torch.zeros((rows, rows), dtype=torch.float64, device="cuda")
            D = torch.zeros_like(P)
            engine.contract(ctx, mode, A, A, tiles, dof, None if mode == engine.MODE_RAW else P, D, prods, e, k_chunk=kc)
            outs.append((P, D))
        torch.cuda.synchronize()
        for P, D in outs[1:]:
            # every chunk's integer sum is exact; only the float64 additions of the scaled chunk
            # sums are ordered differently, so results agree to rounding of the largest partial sum
            scale = float(outs[0][1].abs().max())
            torch.testing.assert_close(D, outs[0][1], rtol=1e-14, atol=1e-14 * scale)
            torch.testing.assert_close(P, outs[0][0], rtol=1e-9, atol=0)


def test_adaptive_schedule_refines_significant_tiles_only():
    """Opt-in adaptive schedule (option "adaptive_min_cells"): tiles run 6 digit products first and
    only tiles holding a pair with r^2 n > 64 are redone with all 8.  Refined tiles equal the full schedule bit for bit, the others
    stay within |dr| <= 1e-7 and rel dP <= 1e-4, and the decision is per tile (any tile subset, the
    rectangular mode and the mirrored tile give the same bits)."""
    rows, n = 3000, 16384
    ctx, p, A, rank, prods = _sliced(rows, n)
    dof = (n - 1 - rank) / 2
    tiles = engine.coex_tiles(rows)

    def run(adaptive, mode=engine.MODE_COEX, tl=tiles):
        engine.set_option("adaptive_min_cells", 8192 if adaptive else 0)
        try:
            P = torch.zeros((rows, rows), dtype=torch.float64, device="cuda")
            D = torch.zeros_like(P)
            engine.contract(ctx, mode, A, A, tl, dof, P, D, prods)
            torch.cuda.synchronize()
            return P, D
        finally:
            engine.set_option("adaptive_min_cells", 0)

    Pf, Df = run(False)
    Pa, Da = run(True)
    refined = engine.last_refined(ctx, len(tiles))
    assert 0 < refined < len(tiles), (refined, len(tiles))
    sd = torch.sqrt(A.var[:, None] * A.var[None, :])
    assert float(((Da - Df).abs() / sd).max()) <= 1e-7
    big = Pf >= 1e-300
    assert float(((Pa - Pf).abs()[big] / Pf[big]).max()) <= 1e-4
    z2 = (Df / sd) ** 2 * n
    hot = (z2 > 64.5) & ~torch.eye(rows, dtype=torch.bool, device="cuda")        # clearly beyond the threshold
    assert bool(hot.any()) and torch.equal(Pa[hot], Pf[hot]) and torch.equal(Da[hot], Df[hot])
    # same decision whatever the launch looks like
    perm = np.random.default_rng(1).permutation(len(tiles))
    P2 = torch.zeros_like(Pa)
    D2 = torch.zeros_like(Pa)
    engine.set_option("adaptive_min_cells", 8192)
    try:
        for chunk in np.array_split(perm, 4):
            engine.contract(ctx, engine.MODE_COEX, A, A, tiles[chunk], dof, P2, D2, prods)
        torch.cuda.synchronize()
    finally:
        engine.set_option("adaptive_min_cells", 0)
    assert torch.equal(P2, Pa) and torch.equal(D2, Da)
    Pr, Gr = run(True, engine.MODE_DE, engine.rect_tiles(rows, rows))
    # (diagonal tiles hold r = 1 in the rectangular mode and are always refined there: compare the others)
    tid = torch.arange(rows, device="cuda") // 128
    off = tid[:, None] != tid[None, :]
    assert torch.equal(Pr[off], Pa[off])
    assert torch.equal(Pr[off], Pr.T[off])                                       # tile (i, j) and tile (j, i) agree


def test_coex_adaptive_against_oracle():
    """End to end with the adaptive schedule switched on: 12,000 cells x 700 genes with planted
    modules (P down to < 1e-300), against the CPU oracle at the BASELINE tolerances."""
    p = synth.host_problem(1009, 700, 12000)
    ref = orc.coex(p["dt"], p["dc"])
    engine.set_option("adaptive_min_cells", 8192)
    try:
        got = norm.coex(p["dt"], p["dc"])
    finally:
        engine.set_option("adaptive_min_cells", 0)
    _check_coex(got, ref)
    iu = np.triu_indices(700, 1)
    assert (ref[0][iu] < 1e-250).sum() > 10 and (ref[0][iu] > 1e-3).sum() > 1000


def test_dynamic_and_static_tile_schedulers_agree():
    """The single-CTA tcgen05 kernel (``umma_pair=0``: co-expression at the default preset would take the
    pair kernel, whose claiming test_contract_pair.py covers) claims tiles from a global counter by default;
    the static round-robin order gives the same bits (few tiles, many tiles, and a tile count below the SM
    count)."""
    for rows, n in ((300, 700), (2500, 2048), (5000, 256)):
        ctx, p, A, rank, prods = _sliced(rows, n)
        dof = (n - 1 - rank) / 2
        outs = []
        try:
            engine.set_option("umma_pair", 0)
            for dyn in (1, 0, 1):
                engine.set_option("umma_dynamic", dyn)
                P = torch.zeros((rows, rows), dtype=torch.float64, device="cuda")
                D = torch.zeros_like(P)
                engine.contract(ctx, engine.MODE_COEX, A, A, engine.coex_tiles(rows), dof, P, D, prods)
                outs.append((P, D))
        finally:
            engine.set_option("umma_dynamic", 1)
            engine.set_option("umma_pair", -1)
        torch.cuda.synchronize()
        for P, D in outs[1:]:
            assert torch.equal(P, outs[0][0]) and torch.equal(D, outs[0][1])


def test_overflow_plan_from_energies():
    rows, n = 300, 3000
    ctx, p, A, rank, prods = _sliced(rows, n)
    assert engine.plan_k_chunk(A, A, prods) == 0
    em = A.energy_max.cpu().numpy()
    ks = engine._lib.load().nsr_cell_splits(n)
    assert (em[:ks, :3] > 0).all() and (em[ks:] == 0).all()
    # exact per-row digit energies can only be below the reported maxima
    sl = A.slices.cpu().numpy().astype(np.int64)
    true_total = (sl ** 2).sum(axis=2).max(axis=1)          # per plane: max over rows of the full-row energy
    assert (true_total <= em.sum(axis=0)[:3] + 1e-6).all()
    # inflate the energies: the planner must fall back to chunks that are provably safe
    big = em * 1e6
    kc = engine.plan_k_chunk(A, A, prods, energies=(big, big))
    assert kc > 0 and kc % 128 == 0


def test_covariate_basis_device_matches_host():
    """nsr_cov_gram / nsr_cov_apply: same basis as the numpy restatement, orthonormal to rounding,
    rank rule of inv_rank (association.py:77), also for rank-deficient and single-row covariates."""
    rng = np.random.default_rng(17)
    ctx = engine.context(0)
    for nc, n, dup in [(1, 77, False), (4, 1000, False), (9, 100_003, True), (40, 5000, True)]:
        dc = rng.normal(size=(nc, n)) * rng.uniform(0.1, 30, size=(nc, 1))
        dc[-1] = 1.0
        if dup and nc > 2:
            dc[1] = 2 * dc[0] - 3 * dc[-1]                 # exact linear dependence
        Qh, rh, Wh = association.covariate_basis(dc)
        Qd, rd, Wd = association.covariate_basis_device(ctx, dc)
        assert rd == rh == (nc - 1 if dup and nc > 2 else nc)
        Qd = Qd.cpu().numpy()
        np.testing.assert_allclose(Qd @ Qd.T, np.eye(rd), atol=1e-13)
        # same subspace: the projectors agree (individual rows may differ by a rotation)
        x = rng.normal(size=(5, n))
        np.testing.assert_allclose((x @ Qd.T) @ Qd, (x @ Qh.T) @ Qh, atol=1e-9)
        np.testing.assert_allclose(Wd @ dc, Qd, atol=1e-8)
    Qd, rd, _ = association.covariate_basis_device(ctx, np.zeros((3, 50)))
    assert Qd is None and rd == 0


def test_residual_planes_reconstruct_projection():
    rng = np.random.default_rng(5)
    x = rng.normal(size=(77, 1000)) + 4
    dc = np.concatenate([rng.normal(size=(3, 1000)), np.ones((1, 1000))])
    Qt, rank, _ = association.covariate_basis(dc)
    ctx = engine.context(0)
    for S in (3, 4):
        A = engine.residualize(ctx, torch.from_numpy(x).cuda(), torch.from_numpy(Qt).cuda(), S)
        z = tl.residual(x, Qt)
        want = tl.hadamard128(z)
        got = engine.unslice(ctx, A).cpu().numpy()
        q = A.quantum.cpu().numpy()
        assert (np.abs(got - want) <= 0.5000001 * q[:, None]).all()
        np.testing.assert_allclose(A.var.cpu().numpy(), (z ** 2).mean(1), rtol=1e-12)
        sl = A.slices.cpu().numpy()
        assert np.abs(sl[0].astype(int)).max() <= 127


def test_pvalue_kernel_known_answers():
    g = load_golden("pvalue_kat")
    ctx = engine.context(0)
    got = engine.pvalue(ctx, torch.from_numpy(g["r2"]).cuda(), g["a"][:, 0]).cpu().numpy()
    assert_p_close(got, g["P"], rtol=1e-9)


# ---- the regime the exact-integer design exists for: 100k cells, P down to 1e-300 ----------
def _planted_loadings(rng, n_gene, lo, hi, n_null):
    """Loadings a_g on one shared factor: r_ij = a_i a_j / sqrt((1+a_i^2)(1+a_j^2))."""
    a = rng.uniform(lo, hi, size=n_gene)
    a[:n_null] = 0.0
    return a


def test_coex_100k_cells_tail():
    """100,000 cells x 300 genes, 9 covariates, planted |r| from ~0.02 to ~0.13: P spans 1 .. < 1e-300.
    At this cell count the P = 1e-300 edge needs |dr| <~ 8e-9 (d ln P / dr ~ n r): the reason the
    contraction is exact-integer.  Against the float64 oracle at the BASELINE tolerances."""
    rng = np.random.default_rng(4100)
    n, g = 100_000, 300
    b = rng.integers(0, 6, size=n)
    dc = np.array([(b == i).astype(float) for i in range(1, 6)] + [rng.normal(size=n) for _ in range(3)] + [np.ones(n)])
    a = _planted_loadings(rng, g, 0.14, 0.38, 60)
    f = rng.normal(size=n)
    dt = rng.normal(size=(g, n))
    dt += a[:, None] * f[None, :]
    dt += 0.3 * dc[5][None, :] + rng.uniform(2, 6, size=(g, 1))            # covariate effect + gene level
    ref = orc.coex(dt, dc)
    got = norm.coex(dt, dc)
    _check_coex(got, ref)
    iu = np.triu_indices(g, 1)
    Pu = ref[0][iu]
    assert ((Pu >= 1e-300) & (Pu <= 1e-200)).sum() >= 50, ((Pu >= 1e-300) & (Pu <= 1e-200)).sum()
    assert (Pu < 1e-300).sum() >= 50 and (Pu > 1e-3).sum() >= 1000
    r = np.abs(pearson_from(ref[1], ref[2], ref[2])[iu])
    assert r.max() > 0.12 and (r < 0.02).sum() > 1000
    # device tensors in: same bits as the host path
    P_d, D_d, v_d = norm.coex(torch.from_numpy(dt).cuda(), torch.from_numpy(dc).cuda())
    assert np.array_equal(P_d.cpu().numpy(), got[0]) and np.array_equal(D_d.cpu().numpy(), got[1])


def test_de_million_cells_tail():
    """1,000,000 cells, binary groupings: P down to 1e-300 needs |r| ~ 0.037 (SURVEY 8c tail point
    r = 0.037 -> 7.19e-300).  de(single=0) against the oracle; cell-chunked int32 accumulation."""
    rng = np.random.default_rng(4101)
    n, g, k = 1_000_000, 40, 8
    dc = np.concatenate([rng.normal(size=(2, n)), np.ones((1, n))])
    dg = (rng.random((k, n)) < 0.01).astype(np.float64)
    dt = rng.normal(size=(g, n)) + 2.0
    eff = np.linspace(0.02, 0.46, g)                       # r = eff * sqrt(p (1 - p)) / sd: up to ~0.045
    for j in range(g):
        dt[j] += eff[j] * dg[j % k]
    ref = orc.de(dg, dt, dc)
    got = norm.de(dg, dt, dc)
    assert_p_close(got[0], ref[0])
    np.testing.assert_allclose(got[3], ref[3], rtol=1e-7)
    np.testing.assert_allclose(got[4], ref[4], rtol=1e-7)
    scale = np.sqrt(ref[4] / ref[3][:, None])
    assert (np.abs(got[1] - ref[1]) <= R_ATOL * scale + 1e-12).all()
    assert ((ref[0] >= 1e-300) & (ref[0] <= 1e-150)).sum() >= 5 and (ref[0] < 1e-300).sum() >= 1


def test_de_single4_config3_shape():
    """BASELINE configs[2] shape with fewer genes: 50,000 cells x 400 genes x 300 gRNAs (Bernoulli 0.02),
    de(single=4): every gRNA tested with the other 299 as covariates (association_test_4,
    association.py:421-576).  The 300 x 300 Gram matrix of the residualised gRNAs is factorised on
    the device (nsr_de4_solve); against the oracle's per-gRNA pseudo-inverses."""
    p = synth.host_problem(1003, 400, 50000, n_group=300, group_p=0.02)
    ref = orc.de(p["dg"], p["dt"], p["dc"], single=4)
    got = norm.de(p["dg"], p["dt"], p["dc"], single=4)
    assert_p_close(got[0], ref[0])
    np.testing.assert_allclose(got[3], ref[3], rtol=1e-7)
    np.testing.assert_allclose(got[4], ref[4], rtol=1e-7)
    scale = np.sqrt(ref[4] / ref[3][:, None])
    assert (np.abs(got[1] - ref[1]) <= R_ATOL * scale + 1e-12).all()
    assert ref[0].min() < 1e-20


@pytest.mark.parametrize("world,gather", [pytest.param(w, False, id=str(w)) for w in (2, 3, 4, 8)] +
                         [pytest.param(w, True, id="%d-gather" % w) for w in (2, 3, 4, 8)])
def test_pairs_schedule_emulated(world, gather):
    """The multi-GPU block-pair schedule, emulated on ONE device: every rank's plan (diagonal block in
    NSR_MODE_COEX_UPPER, block pairs in NSR_MODE_COEX_RECT incl. the split pair at distance world/2)
    is run in turn through the product's own ``parallel.contract_plan`` and assembled with the
    product's own ``parallel.assemble_dense``; the result must equal the single-GPU NSR_MODE_COEX
    matrices bit for bit (ragged last block: 1,900 genes).  Results go ``home`` (the full host matrices)
    or, with ``gather``, the transposed rectangles go into the other ranks' outputs (``coexnet_all_devices``;
    here copies within the one device), after which every rank holds complete rows."""
    from normalisr_b200 import parallel
    n_gene, n = 1900, 3000
    ctx = engine.context(0)
    p = synth.device_problem(1011, n_gene, n, "cuda")
    Qt, crank, _ = association.covariate_basis_device(ctx, p["dc"])
    S, prods = engine.PRESETS["default"]
    dof = (n - 1 - crank) / 2
    full = engine.residualize(ctx, p["dt"], Qt, S)
    P1 = torch.zeros((n_gene, n_gene), dtype=torch.float64, device="cuda")
    D1 = torch.zeros_like(P1)
    engine.contract(ctx, engine.MODE_COEX, full, full, engine.coex_tiles(n_gene), dof, P1, D1, prods)
    blk = parallel.row_split(n_gene, world)
    blocks = [parallel.residualize_block(ctx, p["dt"][r * blk:(r + 1) * blk], Qt, S, blk) for r in range(world)]
    Ps, Ds = [], []
    # `home`: the FULL symmetric host matrices that all ranks fill (rectangles + their transposes, written by
    # the kernel's mirrored stores) - what one caller gets back from the multi-GPU path
    home = (torch.full((n_gene, n_gene), -7.0, dtype=torch.float64).pin_memory(),
            torch.full((n_gene, n_gene), -7.0, dtype=torch.float64).pin_memory())
    outs = [tuple(torch.zeros((parallel.block_rows(n_gene, world, r), n_gene), dtype=torch.float64, device="cuda")
                  for _ in range(2)) for r in range(world)]
    for r in range(world):
        rounds = [(src, parity, blocks[src], []) for _, src, parity in parallel.exchange_plan(world, r)]
        if gather:
            P, D = parallel.contract_plan(ctx, blocks[r], rounds, r, world, n_gene, dof, prods, 0, out=outs[r],
                                          gather=outs, single_launch=(r % 2 == 0))
        else:
            P, D = parallel.contract_plan(ctx, blocks[r], rounds, r, world, n_gene, dof, prods, 0, home=home,
                                          single_launch=(r % 2 == 0))
        Ps.append(P)
        Ds.append(D)
    torch.cuda.synchronize()
    if gather:
        for r in range(world):
            r0 = r * blk
            assert torch.equal(outs[r][0], P1[r0:r0 + outs[r][0].shape[0]])
            assert torch.equal(outs[r][1], D1[r0:r0 + outs[r][1].shape[0]])
    else:
        assert torch.equal(home[0], P1.cpu()) and torch.equal(home[1], D1.cpu())
    assert torch.equal(parallel.assemble_dense(Ps, n_gene, world), P1)
    assert torch.equal(parallel.assemble_dense(Ds, n_gene, world), D1)
    assert torch.equal(torch.cat([b.var[:parallel.block_rows(n_gene, world, r)] for r, b in enumerate(blocks)]), full.var)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs in one process")
def test_all_devices_one_process():
    """``norm.coex(dt, dc, devices=...)`` / ``norm.de(..., devices=...)`` from ONE process on 2+ GPUs: the
    reference's complete return value, bit-identical to the single-GPU call (tools/all_devices_check.py runs
    the same comparison at larger sizes on the multi-GPU boxes)."""
    p = synth.device_problem(1012, 1900, 3000, "cuda")
    dt, dc = p["dt"].cpu().numpy(), p["dc"].cpu().numpy()
    P1, D1, v1 = norm.coex(dt, dc)
    for _ in range(2):
        P, D, v = norm.coex(dt, dc, devices="all")
        assert np.array_equal(P, P1) and np.array_equal(D, D1) and np.array_equal(v, v1)
    dg = (np.random.default_rng(2).random((20, 3000)) < 0.05).astype(np.float64)
    for single in (0, 4):
        r1, rn = norm.de(dg, dt, dc, single=single), norm.de(dg, dt, dc, single=single, devices="all")
        assert all((a is None and b is None) or np.array_equal(a, b) for a, b in zip(r1, rn))


def test_single4_same_golden_and_oracle():
    """single=4 with dy=None (association.py:492-496, 517-556, 1036-1065): one inverse of the residualised Gram
    matrix instead of one pseudo-inverse per pair; reference goldens (incl. alpha, gamma, dimreduce,
    rank-deficient covariates) and a larger oracle case through coex(..., single=4)."""
    g = load_golden("single4_same")
    nx = g["dx"].shape[0]
    iu = np.triu_indices(nx, 1)
    for name, ka in (("lowmem", {}), ("alpha", dict(lowmem=False)), ("gamma", dict(return_dot=False)),
                     ("dimreduce", dict(dimreduce=3))):
        r = association.association_tests(g["dx"], None, g["dc"], single=4, **ka)
        assert_p_close(r[0][iu], g["P_" + name][iu])
        np.testing.assert_allclose(r[0], g["P_" + name], rtol=1e-4, atol=1e-300)
        np.testing.assert_allclose(r[1], g["dot_" + name], rtol=1e-8, atol=1e-11)
        np.testing.assert_allclose(r[4], g["vary_" + name], rtol=1e-9)
        assert r[3] is None and (r[0].diagonal() == 0).all() and (r[4].diagonal() == 1).all()
        if not ka.get("lowmem", True):
            np.testing.assert_allclose(r[2], g["alpha_" + name], rtol=1e-7, atol=1e-10)
    r = association.association_tests(g["dx"], None, g["dc2"], single=4, lowmem=False)
    assert_p_close(r[0][iu], g["P_rankdef"][iu])
    np.testing.assert_allclose(r[2], g["alpha_rankdef"], rtol=1e-7, atol=1e-10)
    rng = np.random.default_rng(77)
    n, nx = 2500, 40
    dc = np.concatenate([rng.normal(size=(3, n)), np.ones((1, n))])
    dx = rng.normal(size=(nx, n)) + rng.normal(size=(nx, 4)) @ rng.normal(size=(4, n))
    want = orc.coex(dx, dc, single=4)
    got = norm.coex(dx, dc, single=4)
    iu = np.triu_indices(nx, 1)
    assert_p_close(got[0][iu], want[0][iu])
    np.testing.assert_allclose(got[1], want[1], rtol=1e-8, atol=1e-11)
    np.testing.assert_allclose(got[2], want[2], rtol=1e-9)
    assert want[0][iu].min() < 1e-50
    dev = association.association_tests(torch.from_numpy(dx).cuda(), None, torch.from_numpy(dc).cuda(), single=4)
    assert dev[0].is_cuda and np.allclose(dev[0].cpu().numpy(), got[0], rtol=1e-12, atol=0)
    with pytest.raises(NotImplementedError):                        # linearly dependent rows
        association.association_tests(np.concatenate([dx, dx[:1] + dx[1:2]]), None, dc, single=4)


def test_split_over_cells_is_bit_identical_for_de():
    """Launches with fewer than two waves of tiles split the cells over work items (tile, part) and add the
    parts' integer sums in a second kernel (option "split_k"): same bits as the one-pass launch for the
    rectangular modes, for general and for exact one-plane groupings, with and without overflow chunks."""
    ctx = engine.context(0)
    n, nx, ny = 40000, 300, 900
    p = synth.device_problem(1021, ny, n, "cuda")
    rng = torch.Generator(device="cuda")
    rng.manual_seed(3)
    dg = (torch.rand((nx, n), generator=rng, device="cuda") < 0.02).to(torch.float64)
    xg = torch.randn((nx, n), generator=rng, device="cuda", dtype=torch.float64) + 0.05 * p["dt"][:nx]
    Qt, crank, _ = association.covariate_basis_device(ctx, p["dc"])
    S, prods = engine.PRESETS["default"]
    B = engine.residualize(ctx, p["dt"], Qt, S)
    A_exact, status = engine.residualize_exact(ctx, dg, Qt)
    assert int(status.item()) == 0
    A_gen = engine.residualize(ctx, xg, Qt, S)
    dof = (n - 1 - crank) / 2
    tiles = engine.rect_tiles(nx, ny)
    for A in (A_exact, A_gen):
        for mode in (engine.MODE_DE, engine.MODE_RAW):
            for kc in (0, 8192):
                outs = []
                for split in (1, 0):
                    engine.set_option("split_k", split)
                    P = torch.zeros((nx, ny), dtype=torch.float64, device="cuda")
                    D = torch.zeros_like(P)
                    engine.contract(ctx, mode, A, B, tiles, dof, None if mode == engine.MODE_RAW else P, D, prods, k_chunk=kc)
                    outs.append((P, D))
                engine.set_option("split_k", 1)
                torch.cuda.synchronize()
                if kc == 0:
                    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
                else:       # sequential chunks add SCALED partial sums: equal to rounding only
                    torch.testing.assert_close(outs[0][1], outs[1][1], rtol=1e-13, atol=1e-13 * float(outs[1][1].abs().max()))
                    torch.testing.assert_close(outs[0][0], outs[1][0], rtol=1e-9, atol=0)
                assert float(outs[0][1].abs().max()) > 0


def test_nonfinite_input_raises():
    """The reference asserts finite outputs (association.py:252-255, 1077): a NaN / Inf in dt must not
    come back as 'not significant'."""
    rng = np.random.default_rng(3)
    dt = rng.normal(size=(40, 500))
    dc = np.ones((1, 500))
    for bad in (np.nan, np.inf):
        x = dt.copy()
        x[7, 123] = bad
        with pytest.raises(AssertionError):
            norm.coex(x, dc)
        with pytest.raises(AssertionError):
            norm.de((rng.random((3, 500)) < 0.3).astype(float), x, dc)
    c = np.ones((2, 500))
    c[1, 5] = np.nan
    with pytest.raises(AssertionError):
        norm.coex(dt, c)


# ---- exact single-plane groupings, device solve of single=4, segmented launch -------------------
def test_exact_groupings_plane():
    """nsr_residualize_exact: binary rows become one int8 plane holding the Hadamard mix of the RAW row
    exactly; var / coef are those of the residual; rows that do not qualify raise the status bits."""
    rng = np.random.default_rng(41)
    n, k = 5000, 37
    dc = np.concatenate([rng.normal(size=(3, n)), np.ones((1, n))])
    dg = (rng.random((k, n)) < 0.03).astype(np.float64)
    dg[3] = (rng.random(n) < 0.5) * 2.0                       # small integers, dense
    Qt, rank, _ = association.covariate_basis(dc)
    ctx = engine.context(0)
    Qd = torch.from_numpy(Qt).cuda()
    A, status = engine.residualize_exact(ctx, torch.from_numpy(dg).cuda(), Qd, keep_coef=True)
    assert int(status.item()) == 0 and A.n_slices == 1
    got = engine.unslice(ctx, A).cpu().numpy()
    np.testing.assert_allclose(got, tl.hadamard128(dg), rtol=0, atol=1e-12)          # exact up to the 1/sqrt(128) scale
    z = tl.residual(dg, Qt)
    np.testing.assert_allclose(A.var.cpu().numpy(), (z ** 2).mean(1), rtol=1e-12)
    np.testing.assert_allclose(A.coef.cpu().numpy(), dg @ Qt.T, rtol=1e-10, atol=1e-12)
    # cross products with residualised genes: exact x -> agrees with float64 to the genes' quantisation error
    dt = rng.normal(size=(200, n)) + 0.4 * dc[0] + 3
    B = engine.residualize(ctx, torch.from_numpy(dt).cuda(), Qd, 3)
    outs = []
    for eng in (engine.ENGINE_UMMA, engine.ENGINE_SIMT):
        G = torch.zeros((k, 200), dtype=torch.float64, device="cuda")
        engine.contract(ctx, engine.MODE_RAW, A, B, engine.rect_tiles(k, 200), 1.0, None, G, 3, eng)
        outs.append(G)
    torch.cuda.synchronize()
    assert torch.equal(outs[0], outs[1])                      # tcgen05 and dp4a engines: same integer sums
    want = z @ tl.residual(dt, Qt).T
    scale = np.sqrt(np.outer((dg ** 2).sum(1), (tl.residual(dt, Qt) ** 2).sum(1)))
    assert (np.abs(outs[0].cpu().numpy() - want) / scale).max() < 2e-8
    # Gram matrix of the raw rows: exact integers
    Gxx = torch.zeros((k, k), dtype=torch.float64, device="cuda")
    engine.contract(ctx, engine.MODE_RAW, A, A, engine.rect_tiles(k, k), 1.0, None, Gxx, 1)
    np.testing.assert_allclose(Gxx.cpu().numpy(), dg @ dg.T, rtol=1e-14, atol=0)      # exact integer sums x (1/sqrt(128))^2
    engine.gram_correct(ctx, Gxx, A.coef)
    np.testing.assert_allclose(Gxx.cpu().numpy(), z @ z.T, rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(engine.gram_f64(ctx, torch.from_numpy(dg).cuda(), A.coef).cpu().numpy(), z @ z.T,
                               rtol=1e-9, atol=1e-9)
    # rows that do not qualify
    _, st = engine.residualize_exact(ctx, torch.from_numpy(dg + 0.3 * (rng.random((k, n)) < 0.01)).cuda(), Qd)
    assert int(st.item()) & 1
    _, st = engine.residualize_exact(ctx, torch.from_numpy(np.round(40 * rng.normal(size=(4, n)))).cuda(), Qd)
    assert int(st.item()) & 1                                                          # mixed values beyond +-127
    batch = np.round(dc[:1] > 0.3).astype(np.float64) + 0.0
    dcb = np.concatenate([dc, batch])                                                  # a grouping that IS a covariate
    Qb = torch.from_numpy(association.covariate_basis(dcb)[0]).cuda()
    _, st = engine.residualize_exact(ctx, torch.from_numpy(batch).cuda(), Qb)
    assert int(st.item()) & 2


@pytest.mark.parametrize("single", [0, 4])
def test_de_general_and_exact_grouping_paths_agree(single):
    """de with the groupings as one exact plane (default for binary dg) and through the general
    3-plane route: both within tolerance of the oracle; continuous groupings take the general route."""
    p = synth.host_problem(1013, 300, 4000, n_group=20, group_p=0.05)
    ref = orc.de(p["dg"], p["dt"], p["dc"], single=single)
    for exact in (True, False):
        got = norm.de(p["dg"], p["dt"], p["dc"], single=single, exact_groupings=exact)
        assert_p_close(got[0], ref[0])
        np.testing.assert_allclose(got[3], ref[3], rtol=1e-7)
        np.testing.assert_allclose(got[4], ref[4], rtol=1e-7)
        scale = np.sqrt(ref[4] / ref[3][:, None])
        assert (np.abs(got[1] - ref[1]) <= R_ATOL * scale + 1e-12).all()
    rng = np.random.default_rng(5)
    dgc = rng.normal(size=(7, 4000)) + 0.2 * p["dc"][5]                # continuous "groupings"
    ref = orc.de(dgc, p["dt"], p["dc"], single=single)
    got = norm.de(dgc, p["dt"], p["dc"], single=single)
    assert_p_close(got[0], ref[0])
    scale = np.sqrt(ref[4] / ref[3][:, None])
    assert (np.abs(got[1] - ref[1]) <= R_ATOL * scale + 1e-12).all()


def test_de4_solve_matches_float64_closed_form():
    """nsr_de4_solve (blocked Cholesky + closed form + P-value on the device) against the float64 torch
    restatement of the same closed form, sizes that cross panel borders; a singular Gram matrix raises bit 1."""
    from normalisr_b200 import single4
    rng = np.random.default_rng(9)
    ctx = engine.context(0)
    for nx, ny, n in ((1, 5, 400), (31, 70, 900), (97, 300, 5000), (300, 1000, 20000)):
        rx = (rng.random((nx, n)) < 0.1) - 0.1 + 0.01 * rng.normal(size=(nx, n))
        ry = rng.normal(size=(ny, n)) + 0.3 * rx[rng.integers(0, nx, size=ny)]
        Gxx, Gxy, yy = rx @ rx.T, rx @ ry.T, (ry ** 2).sum(1)
        dxx, dxy, dyy, rank, w = single4.loo_stats(torch.from_numpy(Gxx), torch.from_numpy(Gxy), torch.from_numpy(yy), n, 2)
        P, gam, vy, vx, wd, st = engine.de4_solve(ctx, torch.from_numpy(Gxx).cuda(), torch.from_numpy(Gxy).cuda(),
                                                  torch.from_numpy(yy).cuda(), n, 2, 0, 1e-8, False)
        assert int(st.item()) == 0
        np.testing.assert_allclose(vx.cpu().numpy(), dxx.numpy(), rtol=1e-9)
        np.testing.assert_allclose(vy.cpu().numpy(), dyy.numpy(), rtol=1e-9)
        np.testing.assert_allclose(gam.cpu().numpy(), (dxy / dxx[:, None]).numpy(), rtol=1e-7, atol=1e-12)
        np.testing.assert_allclose(wd.cpu().numpy(), w.numpy(), rtol=1e-7, atol=1e-12)
        r2 = (dxy * dxy / (dxx[:, None] * dyy)).numpy()
        assert_p_close(P.cpu().numpy(), orc.beta_cdf(1 - r2, (n - 1 - (nx - 1 + 2)) / 2), rtol=1e-6)
    rx[5] = rx[0] + rx[1]
    G = rx @ rx.T
    st = engine.de4_solve(ctx, torch.from_numpy(G).cuda(), torch.from_numpy(rx @ ry.T).cuda(), torch.from_numpy(yy).cuda(),
                          n, 2, 0, 1e-8, False)[5]
    assert int(st.item()) & 1


def test_de_single4_rank_deficient_groupings_fall_back():
    """A grouping that duplicates nothing but is the sum of two others: Cholesky breaks down, the host
    branch (the reference's per-x pseudo-inverse) takes over; the reference itself fails its range
    assert here, so only sanity is checked."""
    p = synth.host_problem(1014, 50, 3000, n_group=6, group_p=0.2)
    dg = p["dg"].copy()
    dg[5] = np.minimum(dg[0] + dg[1], 1.0) * 0 + dg[0] + dg[1]
    try:
        got = norm.de(dg, p["dt"], p["dc"], single=4)
        assert np.isfinite(got[0]).all() and ((got[0] >= 0) & (got[0] <= 1)).all()
    except AssertionError:
        pass            # like the reference (association.py:557)


def test_de_single4_mpc_that_truncates_nothing():
    """single=4 hands method / mpc / qr to inv_rank (association.py:528).  An mpc at least as large as the matrices
    inverted selects the exact SVD and truncates nothing (:64, :78-79): same results as mpc = 0 (golden made by
    the reference with mpc = n_group - 1 + n_cov); a truncating mpc or the randomised SVD is refused."""
    g = load_golden("inv_rank")
    dg, dt, dc = g["de_dg"], g["de_dt"], g["de_dc"]
    for ka in (dict(mpc=dg.shape[0] - 1 + dc.shape[0], method="scipy"), dict(mpc=100, qr=2), dict()):
        P, gamma, _, varg, vart = norm.de(dg, dt, dc, single=4, **ka)
        assert_p_close(P, g["de_P"])
        scale = np.sqrt(g["de_vart"] / g["de_varg"][:, None])
        assert (np.abs(gamma - g["de_gamma"]) <= R_ATOL * scale + 1e-12).all()
        np.testing.assert_allclose(varg, g["de_varg"], rtol=1e-7)
        np.testing.assert_allclose(vart, g["de_vart"], rtol=1e-7)
    for ka in (dict(mpc=3), dict(method="sklearn")):
        with pytest.raises(NotImplementedError):
            norm.de(dg, dt, dc, single=4, **ka)


def test_segments_flags_and_done_counters():
    """nsr_contract_segments with its device-side synchronisation, on one GPU: the remote blocks are
    copied in on a side stream that sets the ready flags afterwards (the launch is already queued),
    and a copy stream waits on the done counters before sending each column block home.  Result:
    bit-identical to the single-launch NSR_MODE_COEX matrices."""
    from normalisr_b200 import parallel
    world, n_gene, n = 4, 2300, 2500
    ctx = engine.context(0)
    p = synth.device_problem(1015, n_gene, n, "cuda")
    Qt, crank, _ = association.covariate_basis_device(ctx, p["dc"])
    S, prods = engine.PRESETS["default"]
    dof = (n - 1 - crank) / 2
    full = engine.residualize(ctx, p["dt"], Qt, S)
    P1 = torch.zeros((n_gene, n_gene), dtype=torch.float64, device="cuda")
    D1 = torch.zeros_like(P1)
    engine.contract(ctx, engine.MODE_COEX, full, full, engine.coex_tiles(n_gene), dof, P1, D1, prods)
    blk = parallel.row_split(n_gene, world)
    nbytes = engine.Sliced.storage_bytes(blk, n, S)
    homes = []
    for r in range(world):
        store = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
        homes.append((store, parallel.residualize_block(ctx, p["dt"][r * blk:(r + 1) * blk], Qt, S, blk, storage=store)))
    torch.cuda.synchronize()
    sync = parallel._sync_words(ctx)
    side = torch.cuda.Stream()
    Ps, Ds = [], []
    for rep in range(2):                    # twice: epochs and monotonic counters
        Ps, Ds = [], []
        for r in range(world):
            sync.epoch += 1
            rows_a = parallel.block_rows(n_gene, world, r)
            rounds, stores = [], []
            for d, (_, src, parity) in enumerate(parallel.exchange_plan(world, r)):
                store = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
                stores.append((store, src))
                work = parallel._FlagWork(None, sync.ready_ptr(d + 1), sync.epoch)
                rounds.append((src, parity, engine.Sliced(blk, n, S, "cuda", storage=store, fresh=False), [work]))
            Ph = torch.full((max(rows_a, 1), n_gene), -1.0, dtype=torch.float64).pin_memory()
            Dh = torch.full((max(rows_a, 1), n_gene), -1.0, dtype=torch.float64).pin_memory()
            # the launch is queued first: it contracts the diagonal block and then waits inside the kernel ...
            P, D = parallel.contract_plan(ctx, homes[r][1], rounds, r, world, n_gene, dof, prods, 0, out_host=(Ph, Dh))
            # ... for the "remote" blocks, which only now start to arrive on the side stream
            with torch.cuda.stream(side):
                for d, (store, src) in enumerate(stores):
                    store.copy_(homes[src][0], non_blocking=True)
                    engine.stream_signal(ctx, sync.ready_ptr(d + 1), sync.epoch, stream=side)
            torch.cuda.synchronize()
            Ps.append(P)
            Ds.append(D)
            m = torch.from_numpy(parallel.owned_tile_mask(n_gene, world, r)).repeat_interleave(128, 0)[:rows_a]
            m = m.repeat_interleave(128, 1)[:, :n_gene]
            assert torch.equal(torch.where(m, Ph[:rows_a], torch.zeros(())), torch.where(m, P[:rows_a].cpu(), torch.zeros(())))
            assert torch.equal(torch.where(m, Dh[:rows_a], torch.zeros(())), torch.where(m, D[:rows_a].cpu(), torch.zeros(())))
    assert torch.equal(parallel.assemble_dense(Ps, n_gene, world), P1)
    assert torch.equal(parallel.assemble_dense(Ds, n_gene, world), D1)

