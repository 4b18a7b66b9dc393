"""Mirror of ``normalisr.binnet`` (reference ``src/normalisr/binnet.py``): P-value co-expression
network -> per-row Benjamini-Hochberg Q-values -> thresholded binary network.  This is the
immediate consumer of ``coex`` (SURVEY 8f-1; reference CLI ``run.binnet``, run.py:313-321): with
P left on the device by ``normalisr_b200.normalisr.coex`` it returns a 1-byte/entry network
instead of shipping 8-byte P-values to the host.

    binnet(net, qcut) -> bool (n_gene, n_gene)         binnet.py:134-170
    binnet(net, qcut, sparse=True) -> the same network in CSR form (an extension)
    bh(pv, weight=None) -> Q-values                    binnet.py:77-131

numpy in -> numpy out, CUDA tensor in -> CUDA tensor out.  The per-row procedure runs in
``nsr_binnet`` (csrc/binnet.cu) and reproduces the reference's booleans bit for bit.  The sparse
form runs the same procedure up to each row's threshold (``nsr_binnet_count``), then compacts the
rows (``nsr_binnet_csr_fill``): 16 B read per entry instead of 8 B read + 1 B written.
"""
import numpy as np
import scipy.sparse
import torch

from . import _lib, engine, hoststage

_ROW_CHUNK_BYTES = 1 << 29


def _is_dev(x):
    return isinstance(x, torch.Tensor) and x.is_cuda


def binnet_rows(ctx, P, qcut, diag0=0, out=None, stats=None):
    """Rows of a P-value matrix (CUDA float64, unit column stride) -> uint8 network rows.
    diag0: column index of row 0's diagonal entry (rows of a row block of a larger matrix).
    stats: CUDA uint64[2] accumulating (edges, rows with entries outside [0, 1])."""
    assert P.is_cuda and P.dtype == torch.float64 and P.dim() == 2 and P.stride(1) == 1
    rows, cols = P.shape
    if out is None:
        out = torch.empty((rows, cols), dtype=torch.uint8, device=P.device)
    assert out.dtype == torch.uint8 and out.shape == P.shape and out.stride(1) == 1
    if stats is None:
        stats = torch.zeros(2, dtype=torch.int64, device=P.device)
    ld = P.stride(0) if rows > 1 else cols
    ldo = out.stride(0) if rows > 1 else cols
    _lib.check(ctx.lib.nsr_binnet(ctx.handle, engine._stream(), P.data_ptr(), rows, cols, ld, int(diag0), float(qcut),
                                  out.data_ptr(), ldo, stats.data_ptr()), "nsr_binnet")
    engine.LAUNCHES += 1
    return out, stats


def csr_rows(ctx, P, qcut, diag0=0, stats=None, D=None):
    """Rows of a P-value matrix (as ``binnet_rows``) -> their network in CSR form on the device:
    (indptr int64 (rows + 1,) from 0, indices, P_e, D_e); indices int32, or int64 from 2^31 edges on.  With
    ``D`` (a matrix like P), P_e and D_e are P and D at the edges, aligned with the indices (else None).
    Waits for the device once (the edge count sizes the arrays); raises AssertionError for values outside
    [0, 1] or not finite."""
    assert P.is_cuda and P.dtype == torch.float64 and P.dim() == 2 and P.stride(1) == 1
    rows, cols = P.shape
    dev = P.device
    if stats is None:
        stats = torch.zeros(2, dtype=torch.int64, device=dev)
    ld = P.stride(0) if rows > 1 else cols
    thr = torch.empty(rows, dtype=torch.float64, device=dev)
    count = torch.empty(rows, dtype=torch.int64, device=dev)
    _lib.check(ctx.lib.nsr_binnet_count(ctx.handle, engine._stream(), P.data_ptr(), rows, cols, ld, int(diag0),
                                        float(qcut), thr.data_ptr(), count.data_ptr(), stats.data_ptr()),
               "nsr_binnet_count")
    engine.LAUNCHES += 1
    indptr = torch.zeros(rows + 1, dtype=torch.int64, device=dev)
    torch.cumsum(count, 0, out=indptr[1:])
    nnz, invalid = (int(x) for x in torch.stack((indptr[-1], stats[1])).cpu())
    if invalid:
        raise AssertionError('net must be finite with values in [0, 1].')
    indices = torch.empty(nnz, dtype=torch.int32 if nnz < 2 ** 31 else torch.int64, device=dev)
    p_e = d_e = None
    ld_d = 0
    if D is not None:
        assert D.shape == P.shape and D.dtype == torch.float64 and D.stride(1) == 1
        p_e = torch.empty(nnz, dtype=torch.float64, device=dev)
        d_e = torch.empty(nnz, dtype=torch.float64, device=dev)
        ld_d = D.stride(0) if rows > 1 else cols
    if nnz == 0:                                      # no row has an edge: nothing to fill
        return indptr, indices, p_e, d_e
    err = torch.zeros(1, dtype=torch.int64, device=dev)
    ptr = lambda t: t.data_ptr() if t is not None else None           # noqa: E731
    _lib.check(ctx.lib.nsr_binnet_csr_fill(ctx.handle, engine._stream(), P.data_ptr(), rows, cols, ld, int(diag0),
                                           thr.data_ptr(), indptr.data_ptr(), indices.data_ptr(),
                                           indices.element_size(), ptr(D), ld_d, ptr(p_e), ptr(d_e), err.data_ptr()),
               "nsr_binnet_csr_fill")
    engine.LAUNCHES += 1
    if int(err.item()):
        raise RuntimeError("nsr_binnet_csr_fill: the edges of a row disagree with its count")
    return indptr, indices, p_e, d_e


def index_dtype(nnz, n):
    """CSR index dtype of scipy and torch for ``nnz`` entries of an n x n matrix: int32 while both fit, else
    int64 (both arrays)."""
    return np.int32 if max(nnz, n) < 2 ** 31 else np.int64


def concat_csr(pieces, n):
    """One host CSR structure of an n x n matrix from row pieces in row order: ``pieces`` = [(indptr, indices,
    *values)], each indptr (rows_k + 1 entries) counted from its own piece's start.  Returns (indptr, indices,
    *values) as numpy arrays, the index arrays with the dtype of ``index_dtype``, the values concatenated."""
    counts = [np.diff(np.asarray(pc[0], dtype=np.int64)) for pc in pieces]
    nnz = sum(int(c.sum()) for c in counts)
    idt = index_dtype(nnz, n)
    indptr = np.zeros(sum(c.size for c in counts) + 1, dtype=idt)
    np.cumsum(np.concatenate(counts) if counts else np.zeros(0, np.int64), out=indptr[1:])
    indices = np.concatenate([np.asarray(pc[1]) for pc in pieces] + [np.zeros(0, idt)]).astype(idt, copy=False)
    vals = [np.concatenate([np.asarray(pc[2 + k]) for pc in pieces]) for k in range(len(pieces[0]) - 2 if pieces else 0)]
    return (indptr, indices, *vals)


def host_csr(n, indptr, indices):
    """scipy csr_matrix (n x n, bool data) of a network's CSR arrays."""
    return scipy.sparse.csr_matrix((np.ones(indices.size, dtype=bool), indices, indptr), shape=(n, n))


def device_net(ctx, P, qcut, sparse, to_host, D=None):
    """Network of a complete (n, n) P-value matrix on the device: dense bool (CUDA tensor, or numpy with
    ``to_host``) or CSR (torch sparse CSR, or scipy csr_matrix).  With ``D`` (CSR only) returns (net, P_e, D_e):
    P and D at the edges.  Raises like ``binnet``."""
    from .association import _outs
    nt = P.shape[0]
    stats = torch.zeros(2, dtype=torch.int64, device=P.device)
    if not sparse:
        out, _ = binnet_rows(ctx, P, qcut, 0, stats=stats)
        edges, invalid = (int(x) for x in stats.cpu())
        if invalid:
            raise AssertionError('net must be finite with values in [0, 1].')
        if edges == 0:
            raise RuntimeError("Empty binary network.")
        out = out.view(torch.bool)
        return _outs((out,))[0] if to_host else out
    indptr, indices, p_e, d_e = csr_rows(ctx, P, qcut, 0, stats, D=D)
    if indices.numel() == 0:
        raise RuntimeError("Empty binary network.")
    tdt = torch.int32 if index_dtype(indices.numel(), nt) == np.int32 else torch.int64
    indptr, indices = indptr.to(tdt), indices.to(tdt)
    if to_host:
        indptr, indices, p_e, d_e = _outs((indptr, indices, p_e, d_e))
        net = host_csr(nt, indptr, indices)
    else:
        net = torch.sparse_csr_tensor(indptr, indices, torch.ones(indices.numel(), dtype=torch.bool, device=P.device),
                                      size=(nt, nt), check_invariants=False)       # canonical by construction
    return net if D is None else (net, p_e, d_e)


def binnet(net, qcut, sparse=False, device=None):
    """Binarizes a P-value co-expression network to a thresholded Q-value network
    (binnet.py:134-170): Q-values per row (diagonal excluded), ``Q <= qcut``; the diagonal is False.
    Raises like the reference: ValueError (shape, qcut), AssertionError (values outside [0, 1] or
    not finite), RuntimeError("Empty binary network.").

    ``sparse=True`` (an extension): the same network in CSR form with bool data - a
    ``scipy.sparse.csr_matrix`` for host input, a ``torch.sparse_csr_tensor`` on the input's device for CUDA
    input; index arrays int32 while the edge count is below 2^31, else int64.  Column indices ascend in every
    row, and the structure equals ``scipy.sparse.csr_matrix(binnet(net, qcut))``.  The dense form stays the
    default: it reads 8 B and writes 1 B per entry, the CSR form reads P twice (16 B) and writes 4 B per
    edge, so it is smaller only for networks with fewer than about one edge in four entries."""
    if net.ndim != 2:
        raise AssertionError('net must be 2-dimensional.')
    nt = net.shape[0]
    if net.shape[1] != nt or nt <= 1:
        raise ValueError('Wrong shape of net or namet.')
    if qcut <= 0 or qcut >= 1:
        raise ValueError('Q-value cutoff must be between 0 and 1.')
    to_host = not _is_dev(net)
    if sparse:
        return _binnet_sparse(net, qcut, to_host, device)
    ctx = engine.context(device if device is not None else (net.device if not to_host else None))
    with torch.cuda.device(ctx.device):
        stats = torch.zeros(2, dtype=torch.int64, device=ctx.device)
        if not to_host:
            Pd = net.to(torch.float64)
            if Pd.stride(1) != 1:
                Pd = Pd.contiguous()
            out, _ = binnet_rows(ctx, Pd, qcut, 0, stats=stats)
        else:
            # rows are independent: stage the host matrix in row chunks
            src = net if isinstance(net, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(net))
            if src.dtype != torch.float64:
                src = src.to(torch.float64)
            out = torch.empty((nt, nt), dtype=torch.uint8, device=ctx.device)
            step = max(1, min(nt, min(_ROW_CHUNK_BYTES, hoststage.STAGE_BYTES) // (8 * nt)))
            blocks = hoststage.RowBlocks(ctx, src, step, tag="binnet")       # pageable P through page-locked slots
            for r0 in range(0, nt, step):
                r1 = min(nt, r0 + step)
                binnet_rows(ctx, blocks.fetch(r0, r1), qcut, r0, out=out[r0:r1], stats=stats)
        edges, invalid = (int(x) for x in stats.cpu())
        if invalid:
            raise AssertionError('net must be finite with values in [0, 1].')
        if edges == 0:
            raise RuntimeError("Empty binary network.")
        out = out.view(torch.bool)
        if to_host:
            from .association import _outs
            return _outs((out,))[0]
        return out


def _binnet_sparse(net, qcut, to_host, device):
    ctx = engine.context(device if device is not None else (net.device if not to_host else None))
    nt = net.shape[0]
    with torch.cuda.device(ctx.device):
        if not to_host:
            Pd = net.to(torch.float64)
            if Pd.stride(1) != 1:
                Pd = Pd.contiguous()
            return device_net(ctx, Pd, qcut, True, False)
        # host input: row chunks as on the dense path, each chunk's CSR piece appended on the host
        src = net if isinstance(net, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(net))
        if src.dtype != torch.float64:
            src = src.to(torch.float64)
        step = max(1, min(nt, min(_ROW_CHUNK_BYTES, hoststage.STAGE_BYTES) // (8 * nt)))
        blocks = hoststage.RowBlocks(ctx, src, step, tag="binnet")
        pieces = []
        for r0 in range(0, nt, step):
            r1 = min(nt, r0 + step)
            indptr, indices, _, _ = csr_rows(ctx, blocks.fetch(r0, r1), qcut, r0)
            pieces.append((indptr.cpu().numpy(), indices.cpu().numpy()))
        indptr, indices = concat_csr(pieces, nt)
        if indices.size == 0:
            raise RuntimeError("Empty binary network.")
        return host_csr(nt, indptr, indices)


def bh(pv, weight=None, device=None):
    """Benjamini-Hochberg Q-values of a vector (binnet.py:77-131): unique P-values, cumulative
    (weighted) counts normalised to 1, q = p / w clipped to [0, 1], running minimum from the top.
    A helper next to ``binnet`` (which does not call it: the row kernel needs no sort); runs on
    the device with torch primitives."""
    to_host = not _is_dev(pv)
    ctx = engine.context(device if device is not None else (pv.device if not to_host else None))
    p = (pv if isinstance(pv, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(pv))).to(ctx.device)
    assert p.dim() == 1 and p.numel() > 0
    assert bool(torch.isfinite(p).all()) and float(p.min()) >= 0 and float(p.max()) <= 1
    if weight is None:
        wt = torch.ones_like(p, dtype=torch.float64)
    else:
        wt = (weight if isinstance(weight, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(weight))).to(
            ctx.device, torch.float64)
        assert wt.shape == p.shape
        assert bool(torch.isfinite(wt).all()) and float(wt.min()) >= 0 and float(wt.max()) > 0
    vals, inv = torch.unique(p, return_inverse=True)
    w = torch.zeros(vals.numel(), dtype=torch.float64, device=ctx.device).index_add_(0, inv, wt)
    w = torch.cumsum(w, 0)
    w = w / w[-1]
    q = vals.to(torch.float64) / w
    q = torch.where(torch.isfinite(q), q, torch.ones_like(q)).clamp_(0, 1)
    q = torch.flip(torch.cummin(torch.flip(q, [0]), 0).values, [0])
    ans = q[inv].to(p.dtype)
    return ans.cpu().numpy() if to_host else ans


def nodiag(d, split=False):
    """Removes the diagonal of a 2-D numpy array (binnet.py:4-33): the rows without their diagonal
    entry, as a list (split) or concatenated."""
    d = np.asarray(d)
    assert d.ndim == 2
    k = min(d.shape)
    rows = [np.concatenate([d[i, :i], d[i, i + 1:]]) if i < k else d[i] for i in range(d.shape[0])]
    return rows if split else np.concatenate(rows)


def rediag(d, fill=0, shape=None):
    """Inverse of ``nodiag(split=False)`` (binnet.py:36-74)."""
    d = np.asarray(d)
    if shape is None:
        t1 = int(np.sqrt(d.size)) + 1
        assert t1 * (t1 - 1) == d.size
        shape = (t1, t1)
    else:
        assert len(shape) == 2 and shape[0] * shape[1] - min(shape) == d.size
    m = np.full(shape, fill, dtype=d.dtype)
    k = min(shape)
    mask = np.ones(shape, dtype=bool)
    mask[np.arange(k), np.arange(k)] = False
    m[mask] = d
    return m
