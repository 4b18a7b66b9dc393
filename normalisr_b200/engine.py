"""Device-level operators of the hot path: thin Python over the C ABI.

PyTorch is used for device memory, streams and (in ``parallel.py``) NCCL only; every
numerical kernel on the path is in ``libnsr_b200.so``.
"""
import ctypes
import functools
import threading

import numpy as np
import torch

from . import _lib
from ._lib import (ENGINE_SIMT, ENGINE_UMMA, MODE_COEX, MODE_COEX_UPPER, MODE_DE, MODE_RAW,  # noqa: F401
                   TILE)

_ctx_lock = threading.Lock()
_contexts = {}
LAUNCHES = 0          # kernels of libnsr_b200.so launched by this process (bench bookkeeping)

# precision presets: (digit planes, digit-pair products kept)
PRESETS = {"fast": (3, 6), "default": (3, 8), "precise": (4, 10)}


class Context:
    """One per device.  Not for concurrent use from several threads."""

    def __init__(self, device):
        if not torch.cuda.is_available():
            raise _lib.NsrError("normalisr_b200 needs a CUDA device (sm_100a); none is visible and "
                                "there is no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.device("cuda", device)
        h = ctypes.c_void_p()
        _lib.check(self.lib.nsr_ctx_create(device, ctypes.byref(h)), "nsr_ctx_create")
        self.handle = h

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.nsr_ctx_destroy(self.handle)
        except Exception:
            pass


def context(device=None):
    if device is None:
        device = torch.cuda.current_device() if torch.cuda.is_available() else 0
    if isinstance(device, torch.device):
        device = device.index if device.index is not None else torch.cuda.current_device()
    with _ctx_lock:
        if device not in _contexts:
            _contexts[device] = Context(device)
        return _contexts[device]


def _stream():
    return torch.cuda.current_stream().cuda_stream


def padded_cells(n):
    return (n + _lib.KBLOCK - 1) // _lib.KBLOCK * _lib.KBLOCK


class Sliced:
    """Residualised rows as int8 digit planes + per-row quantum / variance (device)."""

    def __init__(self, rows, n, n_slices, device, storage=None, fresh=True):
        self.rows, self.n, self.n_slices = rows, n, n_slices
        self.n_pad = padded_cells(n)
        if storage is None:
            self.slices = torch.empty((n_slices, rows, self.n_pad), dtype=torch.int8, device=device)
            self.quantum = torch.empty(rows, dtype=torch.float64, device=device)
            self.var = torch.empty(rows, dtype=torch.float64, device=device)
        else:
            # carve planes | quantum | var out of one uint8 buffer (peer-mapped exchange buffers)
            nb = n_slices * rows * self.n_pad
            assert storage.dtype == torch.uint8 and storage.numel() >= self.storage_bytes(rows, n, n_slices)
            self.slices = storage[:nb].view(torch.int8).view(n_slices, rows, self.n_pad)
            self.quantum = storage[nb:nb + 8 * rows].view(torch.float64)
            self.var = storage[nb + 8 * rows:nb + 16 * rows].view(torch.float64)
        self.coef = None
        # [cell split][plane]: largest per-row sum of squared digits (see nsr_residualize); it travels with
        # the block in the multi-GPU exchange, so every rank can bound its int32 sums without a collective
        ne = _lib.MAX_SPLITS * _lib.MAX_SLICES
        if storage is None:
            self.energy_max = torch.zeros((_lib.MAX_SPLITS, _lib.MAX_SLICES), dtype=torch.float64, device=device)
        else:
            nb = n_slices * rows * self.n_pad + 16 * rows
            self.energy_max = storage[nb:nb + 8 * ne].view(torch.float64).view(_lib.MAX_SPLITS, _lib.MAX_SLICES)
            if fresh:                # a block about to be written here (not a view of one that is being copied in)
                self.energy_max.zero_()

    @property
    def rows_alloc(self):
        return self.slices.shape[1]

    @staticmethod
    def storage_bytes(rows, n, n_slices):
        return n_slices * rows * padded_cells(n) + 16 * rows + 8 * _lib.MAX_SPLITS * _lib.MAX_SLICES


def residualize(ctx, X, Qt, n_slices, out=None, row_offset=0, keep_coef=False):
    """X: (rows, n) float64 CUDA tensor (row stride arbitrary, unit column stride);
    Qt: (rank, n) float64 CUDA tensor with orthonormal rows, or None.
    Writes rows [row_offset, row_offset+rows) of ``out`` (a Sliced) or a fresh one."""
    assert X.is_cuda and X.dtype == torch.float64 and X.dim() == 2 and X.stride(1) == 1
    rows, n = X.shape
    rank = 0 if Qt is None else Qt.shape[0]
    if rank:
        assert Qt.is_cuda and Qt.dtype == torch.float64 and Qt.shape[1] == n and Qt.stride(1) == 1
    if out is None:
        out = Sliced(rows, n, n_slices, X.device)
        row_offset = 0
    if rank > _lib.MAX_RANK:
        # more covariates than the fused kernels stage in shared memory (NSR_MAX_RANK): project with two
        # float64 library GEMMs into a temporary (in row blocks), then quantise that without covariates
        step = max(1, (1 << 28) // max(1, n))
        for r0 in range(0, rows, step):
            xb = X[r0:r0 + step]
            cf = xb @ Qt.T
            residualize(ctx, (xb - cf @ Qt).contiguous(), None, n_slices, out=out, row_offset=row_offset + r0)
            if keep_coef:
                if out.coef is None:
                    out.coef = torch.zeros((out.rows, rank), dtype=torch.float64, device=X.device)
                out.coef[row_offset + r0:row_offset + r0 + xb.shape[0]] = cf
        return out
    assert out.n == n and out.n_slices == n_slices and row_offset + rows <= out.rows
    coef = None
    if keep_coef and rank:
        if out.coef is None:
            out.coef = torch.zeros((out.rows, rank), dtype=torch.float64, device=X.device)
        coef = out.coef[row_offset:row_offset + rows]
    slices = out.slices[:, row_offset:row_offset + rows]
    # a dimension of extent 1 may carry any stride: use the row length for single-row operands
    ldx = X.stride(0) if rows > 1 else n
    ldq = Qt.stride(0) if rank > 1 else n
    st = ctx.lib.nsr_residualize(
        ctx.handle, _stream(), X.data_ptr(), rows, n, ldx,
        Qt.data_ptr() if rank else None, rank, ldq,
        n_slices, slices.data_ptr(), out.rows_alloc, out.n_pad,
        out.quantum[row_offset:].data_ptr(), out.var[row_offset:].data_ptr(),
        coef.data_ptr() if coef is not None else None, out.energy_max.data_ptr())
    _lib.check(st, "nsr_residualize")
    global LAUNCHES
    # pass A (8 covariates per launch, or the sum-of-squares kernel), its finalize, pass B,
    # stats finalize, sparse fix-up pass
    LAUNCHES += ((rank + 7) // 8 if rank else 1) + 4
    return out


def residualize_exact(ctx, X, Qt, keep_coef=False):
    """Rows of small integers (binary groupings) as ONE exact int8 plane (nsr_residualize_exact).
    Returns (Sliced with n_slices = 1, status): status is a device int32 tensor, non-zero when the rows
    do not qualify (not small integers / mostly explained by the covariates) and the plane must not be
    used."""
    assert X.is_cuda and X.dtype == torch.float64 and X.dim() == 2 and X.stride(1) == 1
    rows, n = X.shape
    rank = 0 if Qt is None else Qt.shape[0]
    out = Sliced(rows, n, 1, X.device)
    if keep_coef and rank:
        out.coef = torch.zeros((rows, rank), dtype=torch.float64, device=X.device)
    status = torch.zeros(1, dtype=torch.int32, device=X.device)
    ldx = X.stride(0) if rows > 1 else n
    ldq = Qt.stride(0) if rank > 1 else n
    st = ctx.lib.nsr_residualize_exact(
        ctx.handle, _stream(), X.data_ptr(), rows, n, ldx, Qt.data_ptr() if rank else None, rank, ldq,
        out.slices.data_ptr(), out.rows_alloc, out.n_pad, out.quantum.data_ptr(), out.var.data_ptr(),
        out.coef.data_ptr() if out.coef is not None else None, out.energy_max.data_ptr(), status.data_ptr())
    _lib.check(st, "nsr_residualize_exact")
    global LAUNCHES
    LAUNCHES += ((rank + 15) // 16 if rank else 1) + 3
    return out, status


def unslice(ctx, s):
    out = torch.empty((s.rows, s.n_pad), dtype=torch.float64, device=s.slices.device)
    _lib.check(ctx.lib.nsr_unslice(ctx.handle, _stream(), s.slices.data_ptr(), s.rows, s.rows_alloc,
                                   s.n_pad, s.n_slices, s.quantum.data_ptr(), out.data_ptr()),
               "nsr_unslice")
    return out


def cov_gram(ctx, C):
    """G = C C^T for a (nc, n) CUDA float64 matrix with unit column stride (nsr_cov_gram)."""
    nc, n = C.shape
    G = torch.empty((nc, nc), dtype=torch.float64, device=C.device)
    ldc = C.stride(0) if nc > 1 else n
    _lib.check(ctx.lib.nsr_cov_gram(ctx.handle, _stream(), C.data_ptr(), nc, n, ldc, G.data_ptr()), "nsr_cov_gram")
    global LAUNCHES
    LAUNCHES += 2
    return G


def cov_apply(ctx, M, C):
    """Q = M C, M (rank, nc) numpy or tensor, C (nc, n) CUDA float64 (nsr_cov_apply)."""
    M_d = torch.as_tensor(np.ascontiguousarray(M), dtype=torch.float64).to(C.device) if not isinstance(M, torch.Tensor) \
        else M.to(C.device, torch.float64).contiguous()
    rank, nc = M_d.shape
    n = C.shape[1]
    Q = torch.empty((rank, n), dtype=torch.float64, device=C.device)
    ldc = C.stride(0) if nc > 1 else n
    _lib.check(ctx.lib.nsr_cov_apply(ctx.handle, _stream(), M_d.data_ptr(), rank, nc, C.data_ptr(), n, ldc,
                                     Q.data_ptr(), n), "nsr_cov_apply")
    global LAUNCHES
    LAUNCHES += 1
    return Q


def project_coef(ctx, X, Q):
    """(coef, sumsq): coef = X Q^T (rows, rank) and sumsq = row sums of X^2 (nsr_project_coef).
    X (rows, n), Q (rank, n) CUDA float64 with unit column stride; Q may be None (sumsq only)."""
    rows, n = X.shape
    rank = 0 if Q is None else Q.shape[0]
    coef = torch.empty((rows, max(rank, 1)), dtype=torch.float64, device=X.device)
    sumsq = torch.empty(rows, dtype=torch.float64, device=X.device)
    ldx = X.stride(0) if rows > 1 else n
    ldq = (Q.stride(0) if rank > 1 else n) if rank else n
    _lib.check(ctx.lib.nsr_project_coef(ctx.handle, _stream(), X.data_ptr(), rows, n, ldx,
                                        Q.data_ptr() if rank else None, rank, ldq, coef.data_ptr(), sumsq.data_ptr()),
               "nsr_project_coef")
    global LAUNCHES
    LAUNCHES += ((rank + 15) // 16 if rank else 1) + 1
    return coef[:, :rank], sumsq


def group_stats(ctx, Ys, Cs, goff):
    """out[g, y, :] = [Cs[:, group g] @ Ys[y, group g], sum Ys[y, group g]^2] (nsr_group_stats).
    Ys (genes, m), Cs (nc1, m) CUDA float64, goff (n_groups + 1,) int64 CUDA."""
    genes, m = Ys.shape
    nc1 = Cs.shape[0]
    ng = goff.numel() - 1
    out = torch.empty((ng, genes, nc1 + 1), dtype=torch.float64, device=Ys.device)
    ldy = Ys.stride(0) if genes > 1 else max(m, 1)
    ldc = Cs.stride(0) if nc1 > 1 else max(m, 1)
    _lib.check(ctx.lib.nsr_group_stats(ctx.handle, _stream(), Ys.data_ptr(), genes, ldy,
                                       Cs.data_ptr() if nc1 else None, nc1, ldc, goff.data_ptr(), ng, out.data_ptr()),
               "nsr_group_stats")
    global LAUNCHES
    LAUNCHES += 1
    return out


def sym_pinv(ctx, G, tol=1e-8):
    """(pinv, rank) of a stack (batch, n, n) of symmetric PSD matrices, inv_rank's rule (nsr_sym_pinv)."""
    G = G.contiguous()
    batch, n, _ = G.shape
    out = torch.empty_like(G)
    rank = torch.empty(batch, dtype=torch.int32, device=G.device)
    _lib.check(ctx.lib.nsr_sym_pinv(ctx.handle, _stream(), G.data_ptr(), batch, n, float(tol), out.data_ptr(),
                                    rank.data_ptr()), "nsr_sym_pinv")
    global LAUNCHES
    LAUNCHES += 1
    return out, rank


def single1_finish(ctx, cu, yy_u, st, n_groups, nc, ci, cx, ccx, ns, vx, dof, P, gamma, vy, alpha, col0, flag):
    """Closed form + P-value of de(single=1) for one block of genes (nsr_single1_finish): writes
    columns [col0, col0 + genes) of P / gamma / vy (n_groups, ny) and alpha (n_groups, ny, nc)."""
    genes = cu.shape[0]
    assert cu.is_contiguous() and st.is_contiguous() and yy_u.is_contiguous() and P.is_contiguous()
    assert cu.shape[1] == nc + 1 and st.shape[1] == genes and st.shape[2] == nc + 2 and st.shape[0] >= n_groups
    _lib.check(ctx.lib.nsr_single1_finish(
        ctx.handle, _stream(), cu.data_ptr(), yy_u.data_ptr(), st.data_ptr(), genes, n_groups, nc,
        ci.data_ptr() if nc else None, cx.data_ptr() if nc else None, ccx.data_ptr() if nc else None,
        ns.data_ptr(), vx.data_ptr(), dof.data_ptr(), P.data_ptr(), gamma.data_ptr(), vy.data_ptr(),
        alpha.data_ptr() if alpha is not None else None, P.shape[1], col0, flag.data_ptr()), "nsr_single1_finish")
    global LAUNCHES
    LAUNCHES += 1


@functools.lru_cache(maxsize=64)
def coex_tiles(rows, strip=12):
    """Upper-triangular 128x128 tile list (tile_row <= tile_col), ordered in column strips so
    that the ~148 tiles in flight share few row blocks (L2 reuse of the operand planes)."""
    t = (rows + TILE - 1) // TILE
    out = []
    for js in range(0, t, strip):
        je = min(js + strip, t)
        for i in range(0, je):
            for j in range(max(i, js), je):
                out.append((i, j))
    return np.asarray(out, dtype=np.int32).reshape(-1, 2)


@functools.lru_cache(maxsize=64)
def rect_tiles(rows_a, rows_b, strip=12):
    ta, tb = (rows_a + TILE - 1) // TILE, (rows_b + TILE - 1) // TILE
    out = []
    for js in range(0, tb, strip):
        for i in range(ta):
            for j in range(js, min(js + strip, tb)):
                out.append((i, j))
    return np.asarray(out, dtype=np.int32).reshape(-1, 2)


_INT32_LIMIT = float(2 ** 31 - 1)


def products_of(n_slices, n_products, n_slices_b=None):
    """Kept digit pairs (a, b), 0-based, grouped by weight a + b.  ``n_slices_b`` differs from
    ``n_slices`` when the A operand is a single exact plane (every product kept)."""
    sb = n_slices if n_slices_b is None else n_slices_b
    if sb != n_slices or n_slices == 1:
        assert n_slices == 1 and n_products == sb
        wmax = sb + 1
    else:
        wmax = {(3, 6): 4, (3, 8): 5, (4, 10): 5}[(n_slices, n_products)]
    groups = {}
    for a in range(n_slices):
        for b in range(sb):
            if a + b + 2 <= wmax:
                groups.setdefault(a + b, []).append((a, b))
    return groups


def plan_k_chunk(A, B, n_products, energies=None):
    """Cells per contraction chunk such that no int32 partial sum can overflow, 0 = one pass.

    For a weight group with products (a, b) and any cell range K, Cauchy-Schwarz gives
    |sum_{k in K} sum_(a,b) dA_a[i,k] dB_b[j,k]| <= sum_(a,b) sqrt(EA_a(K) EB_b(K)), E = sum of squared
    digits over K, which the projection reports as maxima over rows per cell split.  Chunks are
    unions of consecutive splits (+1 split of slack because chunk and split borders differ)."""
    if energies is None:
        ea, eb = A.energy_max.cpu().numpy(), (A if B is A else B).energy_max.cpu().numpy()   # one small sync
    else:
        ea, eb = energies
    if not (np.isfinite(ea).all() and np.isfinite(eb).all()):
        # nsr_residualize poisons the report when a row's sum of squares is not finite
        raise AssertionError('Non-finite values (NaN / Inf) in the input matrix or the covariates.')
    ks = _lib.load().nsr_cell_splits(A.n)
    nblk = A.n_pad // _lib.KBLOCK
    groups = products_of(A.n_slices, n_products, B.n_slices)

    ca = np.concatenate([np.zeros((1, ea.shape[1])), np.cumsum(ea[:ks], axis=0)])
    cb = np.concatenate([np.zeros((1, eb.shape[1])), np.cumsum(eb[:ks], axis=0)])

    def worst(width):
        """Largest bound over all windows of ``width`` consecutive splits (clipped at the end)."""
        lo = np.arange(0, max(1, ks - width + 1))
        hi = np.minimum(ks, lo + width)
        sa, sb = ca[hi] - ca[lo], cb[hi] - cb[lo]
        return max(float(sum(np.sqrt(sa[:, a] * sb[:, b]) for a, b in prods).max()) for prods in groups.values())

    if worst(ks) <= _INT32_LIMIT:
        return 0
    blocks_per_split = max(1, nblk // ks)
    # worst(width) grows with width: bisect for the largest m whose windows of m + 1 splits are safe
    lo_m, hi_m = 0, ks - 1
    while lo_m < hi_m:
        mid = (lo_m + hi_m + 1) // 2
        if worst(mid + 1) <= _INT32_LIMIT:
            lo_m = mid
        else:
            hi_m = mid - 1
    if lo_m >= 1:
        return lo_m * blocks_per_split * _lib.KBLOCK
    # even a single split (+ slack) is not provably safe: fall back to the unconditional bound
    # (every digit -128, 4 products per group: 4 * 2^14 * cells < 2^31): 32768 - 128 cells
    return 32768 - _lib.KBLOCK


def contract(ctx, mode, A, B, tiles, dof_a, P, out2, n_products, engine=ENGINE_UMMA, k_chunk=None):
    """Run the contraction + epilogue for ``tiles`` ((k,2) int32 numpy array of tile coords).
    A may be a single exact plane (``residualize_exact``): then every product with B's planes is kept
    and ``n_products`` is ignored."""
    assert A.n == B.n
    if A.n_slices != B.n_slices or A.n_slices == 1:
        assert A.n_slices == 1
        n_products = B.n_slices
    if k_chunk is None:
        k_chunk = plan_k_chunk(A, B, n_products)
    tiles = np.ascontiguousarray(tiles, dtype=np.int32)
    ld = out2.stride(0) if out2.shape[0] > 1 else out2.shape[1]
    assert out2.stride(1) == 1 and (P is None or P.shape == out2.shape and P.stride(1) == 1)
    assert P is None or out2.shape[0] == 1 or P.stride(0) == ld
    st = ctx.lib.nsr_contract_ab(
        ctx.handle, _stream(), engine, mode,
        A.slices.data_ptr(), A.rows, A.rows_alloc, A.n_slices, A.quantum.data_ptr(), A.var.data_ptr(),
        B.slices.data_ptr(), B.rows, B.rows_alloc, B.n_slices, B.quantum.data_ptr(), B.var.data_ptr(),
        A.n, A.n_pad, n_products,
        tiles.ctypes.data, tiles.shape[0], float(dof_a),
        P.data_ptr() if P is not None else None, out2.data_ptr(), ld, int(k_chunk))
    _lib.check(st, "nsr_contract")
    global LAUNCHES
    LAUNCHES += 1 if not k_chunk else -(-A.n_pad // k_chunk)


def contract_segments(ctx, A, segments, tiles, dof_a, P, out2, n_products, k_chunk=0):
    """Everything one GPU owns under the block-pair schedule in ONE persistent launch
    (nsr_contract_segments).  ``segments``: list of dicts with keys B (Sliced), rows_b, col0, diagonal,
    and optionally ready = (uint32 flag tensor element pointer, value), done = pointer, mirror =
    (P pointer, out2 pointer, ld) for the transposed copy; ``tiles``: (k, 3) int32 array of (segment,
    tile_row, tile_col)."""
    assert 1 <= len(segments) <= _lib.MAX_SEGMENTS
    arr = (_lib.Segment * len(segments))()
    for i, sg in enumerate(segments):
        B = sg["B"]
        assert B.n == A.n and B.n_slices == A.n_slices
        arr[i].b_slices = B.slices.data_ptr()
        arr[i].rows_b = int(sg["rows_b"])
        arr[i].rows_alloc_b = B.rows_alloc
        arr[i].quantum_b = B.quantum.data_ptr()
        arr[i].var_b = B.var.data_ptr()
        arr[i].col0 = int(sg["col0"])
        arr[i].diagonal = 1 if sg.get("diagonal") else 0
        ready = sg.get("ready")
        arr[i].ready = ready[0] if ready else None
        arr[i].ready_value = int(ready[1]) & 0xFFFFFFFF if ready else 0
        arr[i].done = sg.get("done")
        mir = sg.get("mirror")
        arr[i].mirror_P, arr[i].mirror_out2, arr[i].ld_mirror = (mir[0], mir[1], int(mir[2])) if mir else (None, None, 0)
    tiles = np.ascontiguousarray(tiles, dtype=np.int32).reshape(-1, 3)
    ld = out2.stride(0) if out2.shape[0] > 1 else out2.shape[1]
    assert out2.stride(1) == 1 and P.shape == out2.shape and P.stride(1) == 1 and (out2.shape[0] == 1 or P.stride(0) == ld)
    st = ctx.lib.nsr_contract_segments(
        ctx.handle, _stream(), A.slices.data_ptr(), A.rows, A.rows_alloc, A.quantum.data_ptr(), A.var.data_ptr(),
        A.n, A.n_pad, A.n_slices, n_products, arr, len(segments), tiles.ctypes.data, tiles.shape[0], float(dof_a),
        P.data_ptr(), out2.data_ptr(), ld, int(k_chunk))
    _lib.check(st, "nsr_contract_segments")
    global LAUNCHES
    LAUNCHES += 1 if not k_chunk else -(-A.n_pad // k_chunk)


def stream_signal(ctx, flag_ptr, value, stream=None):
    """*flag = value once ``stream`` (default: current) reaches this point (no kernel)."""
    st = stream.cuda_stream if stream is not None else _stream()
    _lib.check(ctx.lib.nsr_stream_signal(ctx.handle, st, flag_ptr, int(value) & 0xFFFFFFFF), "nsr_stream_signal")


def stream_wait_geq(ctx, flag_ptr, value, stream=None):
    """``stream`` waits until (int32)(*flag - value) >= 0 (no kernel)."""
    st = stream.cuda_stream if stream is not None else _stream()
    _lib.check(ctx.lib.nsr_stream_wait_geq(ctx.handle, st, flag_ptr, int(value) & 0xFFFFFFFF), "nsr_stream_wait_geq")


def gram_f64(ctx, X, coef):
    """G = X X^T - coef coef^T in float64 (nsr_gram_f64): Gram matrix of the residualised rows."""
    rows, n = X.shape
    rank = 0 if coef is None else coef.shape[1]
    G = torch.empty((rows, rows), dtype=torch.float64, device=X.device)
    cf = coef.contiguous() if rank else None
    ldx = X.stride(0) if rows > 1 else n
    _lib.check(ctx.lib.nsr_gram_f64(ctx.handle, _stream(), X.data_ptr(), rows, n, ldx, cf.data_ptr() if rank else None,
                                    rank, G.data_ptr(), rows), "nsr_gram_f64")
    global LAUNCHES
    LAUNCHES += 3 if rank else 2
    return G


def gram_correct(ctx, G, coef):
    """G = (G + G^T)/2 - coef coef^T in place (nsr_gram_correct)."""
    rows = G.shape[0]
    rank = 0 if coef is None else coef.shape[1]
    if rank == 0:
        return G
    cf = coef.contiguous()
    _lib.check(ctx.lib.nsr_gram_correct(ctx.handle, _stream(), G.data_ptr(), rows, G.stride(0), cf.data_ptr(), rank),
               "nsr_gram_correct")
    global LAUNCHES
    LAUNCHES += 2
    return G


def de4_solve(ctx, Gxx, Gxy, yy, n_cells, rank_c, dimreduce, tol, return_dot):
    """Leave-one-out regression of association_test_4 on the device (nsr_de4_solve).  Gxx is destroyed.
    Returns (P, out2, vary, varx, w, status) - status is a device int32 tensor (see the header)."""
    nx, ny = Gxy.shape
    assert Gxx.is_contiguous() and Gxx.shape == (nx, nx) and Gxy.stride(1) == 1 and yy.is_contiguous()
    dev = Gxy.device
    P = torch.empty((nx, ny), dtype=torch.float64, device=dev)
    out2 = torch.empty_like(P)
    vary = torch.empty_like(P)
    w = torch.empty_like(P)
    varx = torch.empty(nx, dtype=torch.float64, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    ld_xy = Gxy.stride(0) if nx > 1 else ny
    _lib.check(ctx.lib.nsr_de4_solve(ctx.handle, _stream(), Gxx.data_ptr(), nx, Gxy.data_ptr(), ny, ld_xy, yy.data_ptr(),
                                     int(n_cells), int(rank_c), int(dimreduce), float(tol), 1 if return_dot else 0,
                                     P.data_ptr(), out2.data_ptr(), vary.data_ptr(), ny, varx.data_ptr(), w.data_ptr(), ny,
                                     status.data_ptr()), "nsr_de4_solve")
    global LAUNCHES
    LAUNCHES += 3 * ((nx + 31) // 32) + 8
    return P, out2, vary, varx, w, status


def last_refined(ctx, n_tiles):
    """Tiles recomputed with all digit products by the latest adaptive contraction of n_tiles tiles."""
    out = ctypes.c_int64(0)
    _lib.check(ctx.lib.nsr_last_refined(ctx.handle, _stream(), int(n_tiles), ctypes.byref(out)), "nsr_last_refined")
    return int(out.value)


def pvalue(ctx, r2, a):
    """P = I_{1-r2}(a, 1/2); r2 (rows, cols) CUDA float64, a scalar or (rows,) per-row."""
    r2 = r2.contiguous()
    rows, cols = (r2.shape[0], r2.shape[1]) if r2.dim() == 2 else (1, r2.numel())
    a_t = torch.as_tensor(a, dtype=torch.float64, device=r2.device).reshape(-1)
    if a_t.numel() == 1:
        a_t = a_t.expand(rows).contiguous()
    assert a_t.numel() == rows
    P = torch.empty_like(r2)
    _lib.check(ctx.lib.nsr_pvalue(ctx.handle, _stream(), r2.data_ptr(), a_t.data_ptr(), cols,
                                  r2.numel(), P.data_ptr()), "nsr_pvalue")
    return P


def copy_block_to_host(ctx, dst_host, src_dev, r0, r1, c0, c1, stream=None):
    """dst_host[r0:r1, c0:c1] <- src_dev[r0:r1, c0:c1] (both 2-D float64, unit column stride),
    asynchronously on ``stream`` (default: current).  dst_host should be pinned."""
    if r1 <= r0 or c1 <= c0:
        return
    es = 8
    st = stream.cuda_stream if stream is not None else _stream()
    _lib.check(ctx.lib.nsr_copy2d(ctx.handle, st,
                                  dst_host.data_ptr() + (r0 * dst_host.stride(0) + c0) * es, dst_host.stride(0) * es,
                                  src_dev.data_ptr() + (r0 * src_dev.stride(0) + c0) * es, src_dev.stride(0) * es,
                                  (c1 - c0) * es, r1 - r0, 0), "nsr_copy2d")


def copy_rect_to_host(ctx, dst_host, dr0, dc0, src_dev, sr0, sc0, rows, cols, stream=None):
    """dst_host[dr0:dr0+rows, dc0:dc0+cols] <- src_dev[sr0:sr0+rows, sc0:sc0+cols] (2-D float64, unit
    column stride), asynchronously on ``stream`` (default: current)."""
    if rows <= 0 or cols <= 0:
        return
    es = 8
    st = stream.cuda_stream if stream is not None else _stream()
    _lib.check(ctx.lib.nsr_copy2d(ctx.handle, st,
                                  dst_host.data_ptr() + (dr0 * dst_host.stride(0) + dc0) * es, dst_host.stride(0) * es,
                                  src_dev.data_ptr() + (sr0 * src_dev.stride(0) + sc0) * es, src_dev.stride(0) * es,
                                  cols * es, rows, 0), "nsr_copy2d")


def copy_rect_to_peer(ctx, dst_dev, dr0, dc0, src_dev, sr0, sc0, rows, cols, stream=None):
    """dst_dev[dr0:dr0+rows, dc0:dc0+cols] <- src_dev[sr0:sr0+rows, sc0:sc0+cols] (2-D float64, unit column
    stride; src on ctx's device, dst on any GPU of this process), asynchronously on ``stream`` of ctx's device."""
    if rows <= 0 or cols <= 0:
        return
    es = 8
    st = stream.cuda_stream if stream is not None else _stream()
    _lib.check(ctx.lib.nsr_copy2d(ctx.handle, st,
                                  dst_dev.data_ptr() + (dr0 * dst_dev.stride(0) + dc0) * es, dst_dev.stride(0) * es,
                                  src_dev.data_ptr() + (sr0 * src_dev.stride(0) + sc0) * es, src_dev.stride(0) * es,
                                  cols * es, rows, 2), "nsr_copy2d")


def copy_peer(ctx, dst, src, stream=None):
    """dst (contiguous tensor on ctx's device) <- src (contiguous tensor of the same byte size on another
    device of this process), asynchronously on ``stream`` of ctx's device (copy engines, no kernel)."""
    nbytes = dst.numel() * dst.element_size()
    assert dst.is_contiguous() and src.is_contiguous() and nbytes == src.numel() * src.element_size()
    st = stream.cuda_stream if stream is not None else _stream()
    _lib.check(ctx.lib.nsr_copy_peer(ctx.handle, st, dst.data_ptr(), src.data_ptr(), src.device.index, nbytes),
               "nsr_copy_peer")


@functools.lru_cache(maxsize=256)
def coex_strip_tiles(t_begin, t_end, strip=12):
    """Upper-triangular tiles whose tile column lies in [t_begin, t_end), in column sub-strips."""
    out = []
    for js in range(t_begin, t_end, strip):
        je = min(js + strip, t_end)
        for i in range(0, je):
            for j in range(max(i, js), je):
                out.append((i, j))
    return np.asarray(out, dtype=np.int32).reshape(-1, 2)


def set_option(name, value):
    _lib.check(_lib.load().nsr_set_option(name.encode(), int(value)), "nsr_set_option")
