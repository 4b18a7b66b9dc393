"""Which kernel a contraction call runs (csrc/contract_route.h, host-only C++) compiled for the host and checked
on a table of calls: the precedence SIMT > pair > adaptive > split over the cells > one pass, the default pair
kernel for co-expression, and the part count of the split."""
import ctypes
import os
import subprocess

import pytest

from conftest import ROOT

SIMT, ONE_PASS, PAIR, ADAPTIVE, SPLIT_CELLS = range(5)
ENGINE_UMMA, ENGINE_SIMT = 0, 1
COEX, DE, RAW, COEX_UPPER, COEX_RECT = range(5)
PRESETS = {"fast": (3, 3, 4), "default": (3, 3, 5), "precise": (4, 4, 5), "exact": (1, 3, 4)}   # planes A, B; wmax
B200_SMS = 148


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("route") / "libroute.so")
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I", os.path.join(ROOT, "normalisr_b200", "csrc"),
                    os.path.join(ROOT, "tests", "contract_route_shim.cpp"), "-o", out], check=True, env=env)
    lib = ctypes.CDLL(out)
    i, i64 = ctypes.c_int, ctypes.c_int64
    lib.route.argtypes = [i] * 7 + [i64] * 4 + [i, i64] + [i] * 4 + [ctypes.POINTER(i)]
    lib.route.restype = i
    return lib


def call(lib, mode=COEX, rows=20000, cols=None, n=100000, preset="default", k_chunk=0, n_segs=1, seg0_mode=None,
         engine=ENGINE_UMMA, ld=None, umma_pair=-1, adaptive_min_cells=0, split_k=1, umma_kblock=128):
    """(route, parts) of an nsr_contract call over every tile of a rows x cols output (COEX: the upper triangle)."""
    sa, sb, wmax = PRESETS[preset]
    cols = rows if cols is None else cols
    tr, tc = -(-rows // 128), -(-cols // 128)
    n_tiles = tr * (tr + 1) // 2 if mode in (COEX, COEX_UPPER) else tr * tc
    n_pad = -(-n // 128) * 128
    chunk = n_pad if k_chunk == 0 or k_chunk >= n_pad else k_chunk
    slab = rows * (cols if ld is None else ld)
    parts = ctypes.c_int(-1)
    r = lib.route(engine, mode, n_segs, mode if seg0_mode is None else seg0_mode, sa, sb, wmax, n, n_pad, chunk, n_tiles,
                  B200_SMS, slab, umma_pair, adaptive_min_cells, split_k, umma_kblock, ctypes.byref(parts))
    return r, parts.value


CASES = [
    # co-expression: the pair kernel at the default preset only, unless asked for
    ("default preset", dict(), (PAIR, 1)),
    ("default, umma_pair=0", dict(umma_pair=0), (ONE_PASS, 1)),
    ("fast", dict(preset="fast"), (ONE_PASS, 1)),
    ("fast, umma_pair=1", dict(preset="fast", umma_pair=1), (PAIR, 1)),
    ("precise", dict(preset="precise"), (ONE_PASS, 1)),
    ("precise, umma_pair=1", dict(preset="precise", umma_pair=1), (PAIR, 1)),
    ("DE at the default preset", dict(mode=DE), (ONE_PASS, 1)),
    # the pair kernel takes one segment and equal plane counts of at least 3
    ("two segments, umma_pair=1", dict(mode=COEX_RECT, n_segs=2, seg0_mode=COEX_UPPER, umma_pair=1), (ONE_PASS, 1)),
    ("one segment of nsr_contract_segments", dict(mode=COEX_RECT, seg0_mode=COEX_UPPER), (ONE_PASS, 1)),
    ("one segment of nsr_contract_segments, umma_pair=1", dict(mode=COEX_RECT, seg0_mode=COEX_UPPER, umma_pair=1),
     (PAIR, 1)),
    ("1-plane A, umma_pair=1", dict(mode=DE, rows=300, cols=20000, preset="exact", umma_pair=1), (ONE_PASS, 1)),
    # the adaptive schedule: n >= adaptive_min_cells, one pass over the cells
    ("adaptive", dict(rows=3000, n=16384, adaptive_min_cells=8192), (ADAPTIVE, 1)),
    ("adaptive at n = adaptive_min_cells", dict(rows=3000, n=8192, adaptive_min_cells=8192), (ADAPTIVE, 1)),
    ("adaptive, n below it", dict(rows=3000, n=4096, adaptive_min_cells=8192), (PAIR, 1)),
    ("adaptive, forced k_chunk", dict(rows=3000, n=16384, adaptive_min_cells=8192, k_chunk=1024), (ONE_PASS, 1)),
    ("adaptive, umma_pair=1", dict(rows=3000, n=16384, adaptive_min_cells=8192, umma_pair=1), (PAIR, 1)),
    ("adaptive, DE", dict(mode=DE, rows=3000, n=16384, adaptive_min_cells=8192), (ADAPTIVE, 1)),
    ("adaptive, RAW", dict(mode=RAW, rows=3000, n=16384, adaptive_min_cells=8192), (ONE_PASS, 1)),
    ("adaptive, fast", dict(rows=3000, n=16384, adaptive_min_cells=8192, preset="fast"), (ONE_PASS, 1)),
    ("adaptive, 12k cells (coex end to end)", dict(rows=700, n=12000, adaptive_min_cells=8192), (ADAPTIVE, 1)),
    # the split over the cells: DE / RAW, fewer than two waves of tiles, last wave less than 3/4 full
    ("DE, 160 tiles, 1M cells", dict(mode=DE, rows=1280, cols=2048, n=1000000), (SPLIT_CELLS, 4)),
    ("RAW, 160 tiles, 1M cells", dict(mode=RAW, rows=1280, cols=2048, n=1000000), (SPLIT_CELLS, 4)),
    ("DE, 160 tiles, split_k=0", dict(mode=DE, rows=1280, cols=2048, n=1000000, split_k=0), (ONE_PASS, 1)),
    ("DE, 148 tiles", dict(mode=DE, rows=128, cols=148 * 128, n=1000000), (ONE_PASS, 1)),
    ("DE, 237 tiles (1.6 waves)", dict(mode=DE, rows=300, cols=10000, n=50000), (ONE_PASS, 1)),
    ("DE, 296 tiles", dict(mode=DE, rows=128, cols=296 * 128, n=1000000), (ONE_PASS, 1)),
    ("DE, slabs over 1 GiB", dict(mode=DE, rows=1280, cols=2048, n=1000000, ld=40000), (ONE_PASS, 1)),
    ("COEX, 6 tiles, 1M cells", dict(rows=300, n=1000000), (PAIR, 1)),
    ("COEX, 6 tiles, 1M cells, umma_pair=0", dict(rows=300, n=1000000, umma_pair=0), (ONE_PASS, 1)),
    ("COEX_RECT, 6 tiles, 1M cells", dict(mode=COEX_RECT, rows=300, cols=300, n=1000000), (ONE_PASS, 1)),
    ("DE, 24 tiles, 40k cells", dict(mode=DE, rows=300, cols=900, n=40000), (SPLIT_CELLS, 25)),
    ("RAW, 24 tiles, 40k cells, k_chunk 8192", dict(mode=RAW, rows=300, cols=900, n=40000, k_chunk=8192),
     (SPLIT_CELLS, 25)),
    ("DE, 1-plane A, 24 tiles", dict(mode=DE, rows=300, cols=900, n=40000, preset="exact"), (SPLIT_CELLS, 25)),
    ("DE, precise, 24 tiles (64-cell k-blocks)", dict(mode=DE, rows=300, cols=900, n=40000, preset="precise"),
     (SPLIT_CELLS, 25)),
    ("DE, 10 tiles, 4096 cells: at most 1024 cells a part", dict(mode=DE, rows=128, cols=1280, n=4096), (SPLIT_CELLS, 4)),
    ("DE, 10 tiles, 4096 cells, 128-cell chunks", dict(mode=DE, rows=128, cols=1280, n=4096, k_chunk=128),
     (SPLIT_CELLS, 32)),
    ("DE, 10 tiles, 128 cells: one k-block", dict(mode=DE, rows=128, cols=1280, n=128), (ONE_PASS, 1)),
    ("DE, 160 tiles, umma_kblock=64", dict(mode=DE, rows=1280, cols=2048, n=1000000, umma_kblock=64), (SPLIT_CELLS, 4)),
    # the dp4a engine takes every call it is given
    ("SIMT", dict(engine=ENGINE_SIMT), (SIMT, 1)),
    ("SIMT, umma_pair=1", dict(engine=ENGINE_SIMT, umma_pair=1), (SIMT, 1)),
    ("SIMT, DE, 160 tiles", dict(engine=ENGINE_SIMT, mode=DE, rows=1280, cols=2048, n=1000000), (SIMT, 1)),
    # the shapes of test_dynamic_and_static_tile_schedulers_agree: the single-CTA kernel needs umma_pair=0
    ("300 x 700 cells", dict(rows=300, n=700), (PAIR, 1)),
    ("300 x 700 cells, umma_pair=0", dict(rows=300, n=700, umma_pair=0), (ONE_PASS, 1)),
    ("2500 x 2048 cells, umma_pair=0", dict(rows=2500, n=2048, umma_pair=0), (ONE_PASS, 1)),
    ("5000 x 256 cells, umma_pair=0", dict(rows=5000, n=256, umma_pair=0), (ONE_PASS, 1)),
]


@pytest.mark.parametrize("kw,want", [c[1:] for c in CASES], ids=[c[0] for c in CASES])
def test_route(lib, kw, want):
    assert call(lib, **kw) == want
