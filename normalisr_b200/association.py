"""Host-side mirror of ``normalisr.association`` for the hot path (reference
``src/normalisr/association.py``).  Same names, argument order, return tuples and
exceptions as the reference, with the numerics running on the GPU:

    association_tests(dx, dy, dc, bsx, bsy, nth, lowmem, return_dot, single, bs4, **ka)

Inputs may be numpy arrays (results come back as numpy arrays, like the reference) or CUDA
tensors (results stay on the device).  ``bsx/bsy/bs4/nth`` are accepted and ignored: tiling
and parallelism are the GPU's business (reference ``_auto_batchsize``, association.py:731-758).
"""
import logging

import numpy as np
import scipy.linalg
import torch

from . import engine, hoststage
from ._lib import MODE_COEX, MODE_DE, MODE_RAW, ENGINE_UMMA, MAX_RANK

_ROW_CHUNK_BYTES = 1 << 30       # host->device granularity for page-locked host inputs
_STAGED_CHUNK_BYTES = 1 << 28    # ... for pageable ones (they pass through two page-locked slots of this size)
# Streamed co-expression pipeline: row chunks of about _PIPE_CHUNK_BYTES, in multiples of _STRIP_TILES 128-row tiles.
# Small chunks on purpose: the output that becomes final with a chunk can only leave once the chunk's strip is
# contracted, and final output is produced fastest at the end (it grows with the square of the rows seen), so the
# device->host leg trails the host->device leg by about one chunk + one strip.  100k cells x 20k genes, one B200:
# 1.2 GB chunks 330 ms, 0.4 GB 318 ms, 0.2 GB (256 rows) 315 ms per call.
_PIPE_CHUNK_BYTES = 1 << 28
_STRIP_TILES = 2
_TIMELINE = None                 # profiling hook (tools/coex_e2e_profile.py): a list that receives (label, chunk, timing event)


# --------------------------------------------------------------------------------------
# covariates: inv_rank(dc dc^T) -> orthonormal basis              (association.py:4-134, 899-903)
# --------------------------------------------------------------------------------------
def inv_rank(m, tol=1E-8, method='auto', logger=None, mpc=0, qr=0, **ka):
    """Pseudo-inverse and rank by SVD with the reference's rules (association.py:4-134): singular values
    below tol * largest are dropped (:77), ``mpc`` > 0 caps the rank (:78-79, :96-97), ``method`` 'auto' picks
    the exact SVD for matrices up to mpc (or mpc == 0) and the randomised truncated SVD of scikit-learn
    (random_state 0, ``qr`` = QR-normalised power iterations, :81-98) beyond.  Host function: the matrices are
    covariate-sized.  The accelerated paths call it with its defaults (exact branch)."""
    m = np.asarray(m, dtype=np.float64)
    if logger is None:
        logger = logging
    if m.ndim <= 1 or m.shape[-1] != m.shape[-2]:
        raise ValueError('Wrong shape for m.')
    if tol <= 0:
        raise ValueError('tol must be positive.')
    if qr < 0 or int(qr) != qr:
        raise ValueError('qr must be non-negative integer.')
    n = m.shape[-1]
    if method == 'auto':
        if m.ndim > 2 and mpc > 0:
            raise NotImplementedError('No current method supports >2 dimensions with mpc>0.')
        method = 'scipy' if (n <= mpc or mpc == 0) else 'sklearn'
    if method not in ('scipy', 'sklearn'):
        raise ValueError('Unknown method {}'.format(method))
    if m.ndim > 2:
        if method == 'sklearn':
            raise NotImplementedError('Not supporting >2 dimensions for method=sklearn.')
        if mpc > 0:
            raise NotImplementedError('Not supporting >2 dimensions for mpc>0.')
        flat = m.reshape((-1,) + m.shape[-2:])
        res = [inv_rank(x, tol=tol, method='scipy', logger=logger, **ka) for x in flat]
        return (np.array([r[0] for r in res]).reshape(m.shape),
                np.array([r[1] for r in res]).reshape(m.shape[:-2]))
    if method == 'scipy':
        try:
            _, s, vt = scipy.linalg.svd(m, **ka)
        except np.linalg.LinAlgError:
            logger.warning("Default scipy.linalg.svd failed. Falling back to option lapack_driver='gesvd'. "
                           "Expecting much slower computation.")
            _, s, vt = scipy.linalg.svd(m, lapack_driver='gesvd', **ka)
    else:
        from sklearn.utils.extmath import randomized_svd
        kq = {}
        if qr >= 1:
            kq['power_iteration_normalizer'] = 'QR'
        if qr > 1:
            kq['n_iter'] = int(qr)
        k = min(mpc, n) if mpc > 0 else n
        while True:                                   # enough components: grow in steps until the spectrum is covered
            _, s, vt = randomized_svd(m, k, random_state=0, **kq, **ka)
            if k == n or s[-1] <= tol * s[0] or mpc > 0:
                break
            k += min(k, n - k)
    n2 = len(s) - int(np.searchsorted(s[::-1], tol * s[0]))
    if mpc > 0:
        n2 = min(n2, mpc)
    v = vt[:n2]
    return ((v.T / s[:n2]) @ v).T, n2


def _basis_weights(gram, tol):
    """(w0, rank): rows of w0 dc are the eigen-directions of the Gram matrix that the reference's
    inv_rank keeps (singular values >= tol * largest, association.py:77), scaled to unit norm."""
    nc = gram.shape[0]
    _, s, vt = np.linalg.svd(gram)
    rank = nc - int(np.searchsorted(s[::-1], tol * s[0]))
    return vt[:rank] / np.sqrt(s[:rank])[:, None], rank


def _reorthonormalise(g2, w0):
    """q0 = w0 dc is orthonormal up to the 1/sqrt(s) amplification of rounding error; with
    g2 = q0 q0^T = L L^T, Qt = L^-1 q0 is orthonormal to rounding.  Returns (L^-1, W = L^-1 w0)."""
    L = np.linalg.cholesky(g2)
    Linv = scipy.linalg.solve_triangular(L, np.eye(L.shape[0]), lower=True)
    return Linv, Linv @ w0


def covariate_basis(dc, tol=1e-8):
    """Return (Qt, rank, W): Qt (rank, n) has orthonormal rows spanning the part of the row
    space of ``dc`` that the reference keeps (eigenvalues of dc dc^T >= tol * largest), so that
    x - Qt^T (Qt x) equals the reference projection x - dc^T dci dc x.  W (rank, n_cov) maps
    basis coefficients back to covariate coefficients: c = W^T (Qt x)  (needed for alpha).
    Host (numpy) version; the product path uses covariate_basis_device (same factorisation,
    the two products over cells on the GPU)."""
    dc = np.asarray(dc, dtype=np.float64)
    nc, n = dc.shape
    if nc == 0 or not (dc != 0).any():          # association.py:899-903
        return None, 0, np.zeros((0, nc))
    gram = dc @ dc.T
    if not np.isfinite(gram).all():
        raise AssertionError('Non-finite values (NaN / Inf) in the covariates.')
    w0, rank = _basis_weights(gram, tol)
    q0 = w0 @ dc
    Linv, W = _reorthonormalise(q0 @ q0.T, w0)
    return np.ascontiguousarray(Linv @ q0), rank, W


_BASIS_CACHE = {}        # device index -> [(key, result, tensor)]: the bases of the most recent covariate TENSORS
_BASIS_CACHE_LEN = 4


def covariate_basis_device(ctx, dc, tol=1e-8):
    """covariate_basis with the O(nc^2 n) products on the device: returns (Qt_dev, rank, W) with
    Qt_dev a (rank, n) CUDA float64 tensor (None when rank == 0).

    A CUDA tensor that was not modified since the previous call (same storage, shape and torch
    version counter, which every in-place operation bumps) reuses that call's basis: repeated
    coex / de calls with the same covariates skip the two small device->host round trips of the
    factorisation."""
    nc, n = dc.shape
    key = basis_cache_key(ctx, dc, tol)
    if key is not None:
        for hit in _BASIS_CACHE.get(ctx.device.index, ()):
            if hit[0] == key:
                return hit[1]
    res = _covariate_basis_device(ctx, dc, tol)
    if key is not None:
        # holding dc keeps its storage from being reused under the same key
        entries = _BASIS_CACHE.setdefault(ctx.device.index, [])
        entries.insert(0, (key, res, dc))
        del entries[_BASIS_CACHE_LEN:]
    return res


def basis_and_dof(ctx, dc, n, dimreduce):
    """``covariate_basis_device`` and the reference's check that ``n`` cells leave degrees of freedom:
    (Qt_dev, rank, W, dof_a), dof_a the first shape parameter of the P-value's beta function."""
    Qt_dev, rank, W = covariate_basis_device(ctx, dc)
    if n <= rank + dimreduce + 1:
        raise ValueError('Insufficient number of cells: must be greater than degrees of freedom '
                         'removed + covariate + 1.')
    return Qt_dev, rank, W, (n - 1 - rank - dimreduce) / 2


def basis_cache_key(ctx, dc, tol=1e-8, tag=None):
    """Identity of an unmodified CUDA covariate tensor (None for anything else)."""
    if _is_dev(dc) and dc.device == ctx.device:
        return (dc.data_ptr(), dc._version, tuple(dc.shape), tuple(dc.stride()), dc.dtype, float(tol), tag)
    return None


def _covariate_basis_device(ctx, dc, tol):
    nc, n = dc.shape
    if nc == 0:
        return None, 0, np.zeros((0, 0))
    if nc > MAX_RANK:                            # wider than the kernels take: host products
        Qt, rank, W = covariate_basis(_as_host_f64(dc), tol)
        return (torch.from_numpy(Qt).to(ctx.device) if rank else None), rank, W
    if _is_dev(dc):
        dc_d = dc.to(ctx.device, torch.float64)
    else:
        dc_d = torch.from_numpy(np.ascontiguousarray(_as_host_f64(dc), dtype=np.float64)).to(ctx.device)
    if dc_d.stride(1) != 1:
        dc_d = dc_d.contiguous()
    with torch.cuda.device(ctx.device):
        gram = engine.cov_gram(ctx, dc_d).cpu().numpy()
        if not np.isfinite(gram).all():
            raise AssertionError('Non-finite values (NaN / Inf) in the covariates.')
        if not gram.any():                       # all-zero covariates, association.py:899-903
            return None, 0, np.zeros((0, nc))
        w0, rank = _basis_weights(gram, tol)
        q0 = engine.cov_apply(ctx, w0, dc_d)
        Linv, W = _reorthonormalise(engine.cov_gram(ctx, q0).cpu().numpy(), w0)
        return engine.cov_apply(ctx, Linv, q0), rank, W


# --------------------------------------------------------------------------------------
# helpers
# --------------------------------------------------------------------------------------
def _is_dev(x):
    return isinstance(x, torch.Tensor) and x.is_cuda


def _as_host_f64(x):
    if isinstance(x, torch.Tensor):
        x = x.detach().cpu().numpy()
    return np.asarray(x)


def _residualize_any(ctx, x, Qt_dev, n_slices, keep_coef, out=None, row_offset=0):
    """Residualise a (rows, n) matrix that lives on the host (numpy array or CPU tensor, staged
    in row chunks so the copy of chunk i+1 overlaps the kernels of chunk i; pinned memory makes
    the copies asynchronous) or on the device."""
    dev = ctx.device
    if _is_dev(x):
        xd = x.to(torch.float64)
        if xd.stride(1) != 1:
            xd = xd.contiguous()
        return engine.residualize(ctx, xd, Qt_dev, n_slices, out=out, row_offset=row_offset,
                                  keep_coef=keep_coef)
    xh = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x))
    if xh.dtype != torch.float64:
        xh = xh.to(torch.float64)
    rows, n = xh.shape
    if out is None:
        out = engine.Sliced(rows, n, n_slices, dev)
        row_offset = 0
    pageable = not xh.is_pinned()
    chunk = max(1, min(rows, (_STAGED_CHUNK_BYTES if pageable else _ROW_CHUNK_BYTES) // max(1, n * 8)))
    copy_stream = torch.cuda.Stream(device=dev)
    main = torch.cuda.current_stream(dev)
    bufs = [torch.empty((chunk, n), dtype=torch.float64, device=dev) for _ in range(2)]
    stager = hoststage.InputStager(xh, chunk, dev)           # pageable input goes through page-locked slots
    done = [None, None]
    for i, r0 in enumerate(range(0, rows, chunk)):
        r1 = min(r0 + chunk, rows)
        b = bufs[i & 1]
        if done[i & 1] is not None:
            copy_stream.wait_event(done[i & 1])          # buffer free again
        stager.copy_rows(b, r0, r1, copy_stream)
        ready = torch.cuda.Event()
        ready.record(copy_stream)
        main.wait_event(ready)
        engine.residualize(ctx, b[:r1 - r0], Qt_dev, n_slices, out=out, row_offset=row_offset + r0,
                           keep_coef=keep_coef)
        done[i & 1] = torch.cuda.Event()
        done[i & 1].record(main)
    main.synchronize()          # staging buffers are released after this
    return out


def _to_device_f64(ctx, x):
    """Whole matrix on the device as float64 with unit column stride."""
    if _is_dev(x):
        xd = x.to(ctx.device, torch.float64)
    else:
        xh = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x))
        if xh.dtype == torch.float64 and xh.dim() == 2 and xh.stride(1) == 1 and not xh.is_pinned() and xh.numel() >= (1 << 22):
            # a large pageable matrix: through the page-locked slots, in row chunks
            rows, n = xh.shape
            xd = torch.empty((rows, n), dtype=torch.float64, device=ctx.device)
            chunk = max(1, min(rows, _STAGED_CHUNK_BYTES // max(1, n * 8)))
            stager = hoststage.InputStager(xh, chunk, ctx.device)
            st = torch.cuda.current_stream(ctx.device)
            for r0 in range(0, rows, chunk):
                stager.copy_rows(xd[r0:], r0, min(rows, r0 + chunk), st)
            st.synchronize()
            return xd
        xd = xh.to(ctx.device, torch.float64, non_blocking=True)
    return xd if xd.stride(1) == 1 else xd.contiguous()


def _residualize_groupings(ctx, dx, Qt_dev, n_slices, keep_coef, exact=True):
    """The x operand of de (groupings / gRNA indicators, de.py:4-132): rows of small integers become ONE
    exact int8 plane of the raw row (nsr_residualize_exact) - the contraction then needs 3 digit products
    instead of 8 and is exact in x; anything else takes the general route.  Returns (Sliced, raw device
    matrix)."""
    xd = _to_device_f64(ctx, dx)
    if exact and (Qt_dev is None or Qt_dev.shape[0] <= MAX_RANK):
        A, status = engine.residualize_exact(ctx, xd, Qt_dev, keep_coef=keep_coef)
        if int(status.item()) == 0:
            return A, xd
    return engine.residualize(ctx, xd, Qt_dev, n_slices, keep_coef=keep_coef), xd


def _mark(label, chunk, stream):
    if _TIMELINE is not None:
        ev = torch.cuda.Event(enable_timing=True)
        ev.record(stream)
        _TIMELINE.append((label, chunk, ev))


def _coex_host_pipeline(ctx, xh, Qt_dev, n_slices, n_products, dof_a, eng, keep_coef, out_host, into=None):
    """Co-expression of a HOST matrix with the three legs overlapped:
      copy stream : chunk c+1 of the expression matrix, host -> device
      main stream : projection of chunk c, then every output tile whose columns lie in chunk c
                    (such a tile only needs rows <= its column, i.e. chunks 0..c)
      d2h stream  : the blocks of P / dot that became final with chunk c, device -> host
    After strip c the square [0, end_c)^2 is complete (mirrored entries included), so the newly
    final part is the column block [0:end_c, begin_c:end_c] plus the row block
    [begin_c:end_c, 0:begin_c].  Returns (A, P_dev, dot_dev).

    ``into`` = (A, P, D): the diagonal block of a multi-GPU job (``parallel``): project into the rank's own Sliced
    block and write the (rows, rows) square into the given views of the rank's output rows (``out_host``: the
    matching views of the job's host matrices).  Nothing waits for the device then: the int32 bound is the caller's
    to verify with the other blocks' energies, and the function returns (A, P, D, event) with the event recorded
    behind the last device->host copy."""
    dev = ctx.device
    rows, n = xh.shape
    if into is None:
        A = engine.Sliced(rows, n, n_slices, dev)
        P = torch.empty((rows, rows), dtype=torch.float64, device=dev)
        D = torch.empty((rows, rows), dtype=torch.float64, device=dev)
    else:
        A, P, D = into
    strip_rows = _STRIP_TILES * engine.TILE
    base = max(strip_rows, (_PIPE_CHUNK_BYTES // max(1, n * 8)) // strip_rows * strip_rows)
    # row chunks: `base` rows while plenty remain, then geometrically smaller ones, so that the work
    # left after the last host->device copy (the last strip's tiles and its device->host copy) is small
    bounds = [0]
    while bounds[-1] < rows:
        left = rows - bounds[-1]
        step = base if left > 3 * base else max(2 * engine.TILE, (left // 3) // engine.TILE * engine.TILE)
        bounds.append(min(rows, bounds[-1] + step))
    chunk = min(base, (rows + engine.TILE - 1) // engine.TILE * engine.TILE)
    copy_stream = torch.cuda.Stream(device=dev)
    d2h_stream = torch.cuda.Stream(device=dev)
    main = torch.cuda.current_stream(dev)
    bufs = [torch.empty((min(chunk, rows), n), dtype=torch.float64, device=dev) for _ in range(2)]
    stager = hoststage.InputStager(xh, min(chunk, rows), dev)
    # results into ordinary (pageable) host matrices leave through a ring of page-locked slots and a worker thread
    drain = None
    if out_host is not None and not all(t.is_pinned() for t in out_host):
        widest = max(bounds[i + 1] - bounds[i] for i in range(len(bounds) - 1))
        drain = hoststage.OutputDrain(ctx, 4 * 8 * rows * widest)
    done = [None, None]
    for i in range(len(bounds) - 1):
        r0, r1 = bounds[i], bounds[i + 1]
        b = bufs[i & 1]
        if done[i & 1] is not None:
            copy_stream.wait_event(done[i & 1])
        _mark("h2d_begin", i, copy_stream)
        stager.copy_rows(b, r0, r1, copy_stream)
        ready = torch.cuda.Event()
        ready.record(copy_stream)
        _mark("h2d_end", i, copy_stream)
        main.wait_event(ready)
        engine.residualize(ctx, b[:r1 - r0], Qt_dev, n_slices, out=A, row_offset=r0, keep_coef=keep_coef)
        done[i & 1] = torch.cuda.Event()
        done[i & 1].record(main)
        _mark("projected", i, main)
        t1 = (r1 + engine.TILE - 1) // engine.TILE
        tiles = engine.upper_tiles(0, t1, r0 // engine.TILE, t1)
        # optimistic single pass over the cells (planning would need a device->host sync per chunk
        # and stall the copy stream); the int32 bound is verified once at the end
        engine.contract(ctx, MODE_COEX, A, A, tiles, dof_a, P, D, n_products, eng, k_chunk=0)
        _mark("contracted", i, main)
        if out_host is not None:
            fin = torch.cuda.Event()
            fin.record(main)
            d2h_stream.wait_event(fin)
            if drain is not None:
                drain.send(d2h_stream, [(dst[a0:a1, b0:b1], src[a0:a1, b0:b1]) for dst, src in zip(out_host, (P, D))
                                        for a0, a1, b0, b1 in ((0, r1, r0, r1), (r0, r1, 0, r0))])
            else:
                for dst, src in zip(out_host, (P, D)):
                    engine.copy_block_to_host(ctx, dst, src, 0, r1, r0, r1, d2h_stream)
                    engine.copy_block_to_host(ctx, dst, src, r0, r1, 0, r0, d2h_stream)
            _mark("d2h_end", i, d2h_stream)
    if drain is not None:
        drain.close()
    if into is not None:
        main.wait_stream(copy_stream)          # the staging buffers go back to the allocator of this stream
        tail = torch.cuda.Event()
        tail.record(d2h_stream)
        return A, P, D, tail
    main.synchronize()
    d2h_stream.synchronize()
    k_chunk = engine.plan_k_chunk(A, A, n_products)
    if k_chunk:
        # some int32 partial sum was not provably exact: redo the contraction in cell chunks
        engine.contract(ctx, MODE_COEX, A, A, engine.coex_tiles(rows), dof_a, P, D, n_products, eng, k_chunk=k_chunk)
        if out_host is not None:
            for dst, src in zip(out_host, (P, D)):
                dst.copy_(src, non_blocking=True)
        main.synchronize()
    return A, P, D


_PINNED_OUT_BYTES = 1 << 30     # results up to this size come back through page-locked staging


def _outs(tensors, host_bufs=None):
    """Device results -> numpy arrays with ONE wait: every tensor is copied asynchronously into page-locked host
    memory (the caller's buffer where one was given, else a block from torch's caching host allocator, which the
    returned array keeps alive) and the stream is synchronised once.  A pageable destination costs a staged copy
    and a page fault per 4 KB of fresh memory: 32 ms for the 72 MB of a 300 x 10,000 de() result against 1.4 ms."""
    host_bufs = list(host_bufs) if host_bufs is not None else []
    host_bufs += [None] * (len(tensors) - len(host_bufs))
    total = sum(t.numel() * t.element_size() for t in tensors if t is not None)
    outs = []
    for t, hb in zip(tensors, host_bufs):
        if t is None:
            outs.append(None)
            continue
        if hb is None:
            hb = torch.empty(t.shape, dtype=t.dtype, pin_memory=total <= _PINNED_OUT_BYTES)
        hb.copy_(t, non_blocking=True)
        outs.append(hb)
    torch.cuda.current_stream().synchronize()
    return tuple(None if h is None else h.numpy() for h in outs)


# --------------------------------------------------------------------------------------
# association_tests                                              (association.py:761-1093)
# --------------------------------------------------------------------------------------
def association_tests(dx, dy, dc, bsx=0, bsy=0, nth=1, lowmem=True, return_dot=True, single=0,
                      bs4=500, **ka):
    """Association tests between all pairs of rows of dx and dy (or within dx when
    ``dy is None``) given covariates dc.  See the reference docstring
    (association.py:772-843) for the model; returns ``(P, dot|gamma, alpha|None, varx|None,
    vary)`` with the reference's shapes.

    Extra keyword arguments understood here (all optional, none changes results beyond the
    stated tolerance): ``precision`` in {'fast','default','precise'}, ``device``,
    ``out`` = (P, dot) preallocated (pinned) CPU tensors that receive the two matrices,
    ``devices`` = "all" | count | list of CUDA devices: host inputs are spread over those GPUs from this
    one process and the caller gets the reference's complete return value (``parallel.coex_all_devices``
    for dy=None, ``parallel.de_all_devices`` otherwise), ``engine`` (tests only)."""
    precision = ka.pop('precision', 'default')
    exact_groupings = ka.pop('exact_groupings', True)
    device = ka.pop('device', None)
    eng = ka.pop('engine', ENGINE_UMMA)
    out_host = ka.pop('out', None)          # optional (P, dot|gamma) host tensors to fill
    devices = ka.pop('devices', None)       # "all" / count / list: every listed GPU of the box, one process
    dimreduce = ka.pop('dimreduce', 0)
    if single not in (0, 1, 4, 5):
        raise ValueError('Unknown value single={}'.format(single))
    if single == 5:
        raise NotImplementedError('normalisr_b200 accelerates single=0, 1 and 4; single=5 ("under '
                                  'development" upstream) is outside the hot path (SURVEY.md 8f).')
    if np.ndim(dimreduce) != 0:
        # the reference's scalar comparison at association.py:213 raises for arrays as well
        raise ValueError('dimreduce must be a scalar.')
    dimreduce = int(dimreduce)
    samexy = dy is None
    if len(dx.shape) != 2 or (not samexy and len(dy.shape) != 2) or len(dc.shape) != 2:
        raise ValueError('Incorrect dx/dy/dc size.')
    n = dx.shape[1]
    if (not samexy and dy.shape[1] != n) or dc.shape[1] != n:
        raise ValueError('Unmatching dx/dy/dc dimensions.')
    if devices is not None:
        from . import parallel
        devs = parallel.visible_devices(devices)
        if len(devs) > 1:
            if _is_dev(dx) or _is_dev(dy) or device is not None:
                raise ValueError('devices= takes host inputs (the matrices are spread over the GPUs).')
            common = dict(precision=precision, dimreduce=dimreduce)
            if not samexy:
                return parallel.de_all_devices(dx, dy, dc, devs, lowmem=lowmem, return_dot=return_dot, single=single,
                                               engine=eng, exact_groupings=exact_groupings, **common, **ka)
            if single != 0 or not (lowmem and return_dot) or ka:
                raise NotImplementedError('devices= with dy=None covers the coex call: single=0, lowmem=True, '
                                          'return_dot=True.')
            P, D, var = parallel.coex_all_devices(dx, dc, devs, out=out_host, **common)
            return (P, D, None, None, var)
        device = devs[0]
    if single == 1:
        from .single1 import association_tests_single1
        if samexy:
            raise NotImplementedError('dy=None with single=1')                # association.py:911-912
        return association_tests_single1(dx, dy, dc, lowmem=lowmem, return_dot=return_dot,
                                         dimreduce=dimreduce, device=device, **ka)
    if single == 4:
        from .single4 import association_tests_single4, association_tests_single4_same
        if samexy:                                                               # association.py:492-496
            return association_tests_single4_same(dx, dc, lowmem=lowmem, return_dot=return_dot, dimreduce=dimreduce,
                                                  device=device, **ka)
        return association_tests_single4(dx, dy, dc, lowmem=lowmem, return_dot=return_dot,
                                         dimreduce=dimreduce, precision=precision, device=device,
                                         engine=eng, exact_groupings=exact_groupings, **ka)
    if ka:
        raise TypeError("association_test_1() got an unexpected keyword argument '{}'".format(
            next(iter(ka))))
    to_host = not _is_dev(dx)
    ctx = engine.context(device if device is not None else (dx.device if _is_dev(dx) else None))
    n_slices, n_products = engine.PRESETS[precision]
    nc = dc.shape[0]
    if nc == 0:
        logging.warning('No covariate dc input.')
    Qt_dev, rank, W, dof_a = basis_and_dof(ctx, dc, n, dimreduce)
    with torch.cuda.device(ctx.device):
        keep_coef = not lowmem
        piped = samexy and to_host
        if piped:
            xh = dx if isinstance(dx, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(dx))
            if xh.dtype != torch.float64:
                xh = xh.to(torch.float64)
            direct = out_host if (out_host is not None and lowmem and return_dot) else None
            if direct is None and out_host is None and lowmem and return_dot:
                # the caller gets fresh (pageable) matrices, like from the reference; they are filled block by
                # block while the pipeline runs
                direct = (torch.empty((dx.shape[0], dx.shape[0]), dtype=torch.float64),
                          torch.empty((dx.shape[0], dx.shape[0]), dtype=torch.float64))
            A, P, out2 = _coex_host_pipeline(ctx, xh, Qt_dev, n_slices, n_products, dof_a, eng, keep_coef,
                                             direct)
            B = A
            if direct is not None:       # P and dot are already in the caller's host buffers
                var_h = A.var.cpu().numpy()
                return (direct[0].numpy(), direct[1].numpy(), None, None, var_h)
        elif samexy:
            A = B = _residualize_any(ctx, dx, Qt_dev, n_slices, keep_coef)
        else:
            A, _ = _residualize_groupings(ctx, dx, Qt_dev, n_slices, keep_coef, exact=exact_groupings)
            B = _residualize_any(ctx, dy, Qt_dev, n_slices, keep_coef)
        nx, ny = A.rows, B.rows
        if not piped:
            P = torch.empty((nx, ny), dtype=torch.float64, device=ctx.device)
            out2 = torch.empty((nx, ny), dtype=torch.float64, device=ctx.device)
        if samexy:
            if not piped:
                engine.contract(ctx, MODE_COEX, A, A, engine.coex_tiles(nx), dof_a, P, out2, n_products, eng)
            gamma = None
            if not (lowmem and return_dot):
                gamma = out2 / A.var[:, None]
        else:
            engine.contract(ctx, MODE_DE, A, B, engine.rect_tiles(nx, ny), dof_a, P, out2,
                            n_products, eng)
            gamma = out2
        alpha = None if lowmem else _alpha(A, B, gamma, W, rank, nc, samexy)
        if samexy and not return_dot:                      # association.py:1058-1061
            out2 = gamma
        elif not samexy and return_dot:                    # association.py:1044-1048
            out2 = gamma * A.var[:, None]
        varx = None if samexy else A.var
        res = (P, out2, alpha, varx, B.var)
        if to_host:
            res = _outs(res, out_host)
    return res


def _alpha(A, B, gamma, W, rank, nc, samexy):
    """alpha[x, y, :] = c_y - gamma[x, y] c_x   (association.py:238-245); for dy=None the
    reference keeps the upper triangle and mirrors it (association.py:1062-1065), which leaves
    a zero diagonal because gamma[x, x] = 1 there."""
    dev = A.var.device
    nx, ny = A.rows, B.rows
    if rank == 0:
        return torch.zeros((nx, ny, nc), dtype=torch.float64, device=dev)
    Wd = torch.from_numpy(W).to(dev)                        # (rank, nc)
    cx = A.coef @ Wd
    cy = B.coef @ Wd
    al = cy[None, :, :] - gamma[:, :, None] * cx[:, None, :]
    if samexy:
        al = torch.triu(al.permute(2, 0, 1), 1)
        al = (al + al.transpose(1, 2)).permute(1, 2, 0).contiguous()
    return al
