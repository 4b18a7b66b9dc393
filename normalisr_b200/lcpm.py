"""``normalisr.lcpm.lcpm`` on the GPU (reference src/normalisr/lcpm.py:21-208; SURVEY 8f-4):
Bayesian logCPM of a read-count matrix, the posterior mean digamma(1 + reads) - digamma(total + 2)
normalised per cell to log counts per million, plus the three cellular covariates (log total
reads, number of zero-count genes, its square), and optionally the reference's posterior
resampling (``varscale != 0``).

Streaming passes over the counts: ``nsr_lcpm_scan`` (min / max / total in one read: the negativity
check, the table length and the total), ``nsr_lcpm_colstats`` (per-cell sums; a pure table gather
without resampling) and ``nsr_lcpm_apply`` (gather + shift).  The digamma / trigamma look-up tables
over the count values (the reference builds the same tables) come from ``torch.special`` on the
device.  numpy in -> numpy out, CUDA tensors in -> CUDA tensors out.

Resampling draws one standard normal deviate per entry.  For numpy input they come from numpy's
global generator exactly as in the reference (``numpy.random.seed(seed)`` when a seed is given, then
one ``numpy.random.randn(n_gene, n_cell)``), so the result is the reference's, deviate for deviate;
for CUDA input they are generated on the device by Philox4x32-10 keyed by ``seed`` (a fresh random
key when ``seed`` is None) with the entry's index as counter - same distribution, another stream;
``noise=`` (a matrix of deviates) overrides both.

Sparse counts - scipy.sparse matrices or arrays (CSR, CSC, COO; integer or float values; int32 or int64 indices) on
the host, torch sparse CSR / CSC / COO tensors on a CUDA device - are never expanded to genes x cells: their index
and value arrays are shipped as they are (host arrays through the page-locked slots), put into canonical CSR on the
device (sorted and duplicates summed only when needed; O(nnz)) and read by ``nsr_lcpm_colstats_csr`` /
``nsr_lcpm_apply_csr``, which expand 64 genes x 256 cells at a time in shared memory and run the dense kernels'
per-cell loops on them.  The result is bit for bit the dense path's on ``reads.toarray()`` (host) /
``reads.to_dense()`` (CUDA): duplicates are summed in the value dtype, floats truncated to integers, and a
non-finite value raises the ValueError of a negative count."""
import logging

import numpy as np
import torch

from . import _lib, engine, hoststage

_ROW_CHUNK_BYTES = 1 << 30
_HOLD_BYTES = 1 << 35          # host counts up to this size are copied to the device once for both passes


def _is_dev(x):
    return isinstance(x, torch.Tensor) and x.is_cuda


_TABLE_LEN = 4096
_TABLES = {}


def _tables(dev):
    """(digamma(1 + c), exp(digamma(1 + c))) for c < 4096 on ``dev``."""
    key = torch.device(dev).index
    if key not in _TABLES:
        lut = torch.special.digamma(torch.arange(1, _TABLE_LEN + 1, dtype=torch.float64, device=dev)).contiguous()
        _TABLES[key] = (lut, torch.exp(lut).contiguous())
    return _TABLES[key]


def _trigamma(x):
    """polygamma(1, x) for x >= 1 to float64 rounding: 15 recurrence steps, then the asymptotic series up to
    B14 at x + 15 (torch.special.polygamma stops at B6 after 6 steps: 5e-10 relative, visible in the
    resampled values at the golden tolerance)."""
    s = torch.zeros_like(x)
    for i in range(15):
        s = s + 1.0 / ((x + i) * (x + i))
    iy = 1.0 / (x + 15.0)
    i2 = iy * iy
    ser = i2 * (1 / 6 + i2 * (-1 / 30 + i2 * (1 / 42 + i2 * (-1 / 30 + i2 * (5 / 66 + i2 * (-691 / 2730 + i2 * (7 / 6)))))))
    return s + iy * (1.0 + 0.5 * iy + ser)


def _sparse_parts(reads):
    """(format, a, b, values) of a sparse count matrix, the caller's own arrays: 'csr' (a = row pointers over genes,
    b = cell indices), 'csc' (a = column pointers over cells, b = gene indices) or 'coo' (a = gene indices, b = cell
    indices).  None for a strided matrix."""
    if isinstance(reads, torch.Tensor):
        if reads.layout == torch.sparse_csr:
            return 'csr', reads.crow_indices(), reads.col_indices(), reads.values()
        if reads.layout == torch.sparse_csc:
            return 'csc', reads.ccol_indices(), reads.row_indices(), reads.values()
        if reads.layout == torch.sparse_coo:
            ij = reads._indices()                           # duplicates allowed: they are summed below
            return 'coo', ij[0], ij[1], reads._values()
        return None
    if not hasattr(reads, 'tocoo'):
        return None
    import scipy.sparse
    if not scipy.sparse.issparse(reads):
        return None
    if reads.format in ('csr', 'csc'):
        nnz = int(reads.indptr[-1])
        return reads.format, reads.indptr, reads.indices[:nnz], reads.data[:nnz]
    coo = reads if reads.format == 'coo' else reads.tocoo()
    return 'coo', coo.row, coo.col, coo.data


def _ship(ctx, x):
    """A host index or value array -> device, through the page-locked slots; unsigned integers travel as the
    signed type of their width, booleans as bytes (undone on the device)."""
    x = np.ascontiguousarray(x)
    if x.dtype.kind == 'u' and x.dtype.itemsize > 1:
        x = x.view('i%d' % x.dtype.itemsize)
    elif x.dtype.kind == 'b':
        x = x.view(np.uint8)
    return hoststage.to_device(ctx, torch.from_numpy(x), tag="lcpm-in")


def _sum_runs(v, starts, nnz):
    """Sums of the runs of equal keys beginning at ``starts`` (v sorted stably by key), each in storage order and in
    v's dtype, as ``toarray()`` adds duplicates."""
    lens = torch.diff(starts, append=torch.tensor([nnz], dtype=starts.dtype, device=starts.device))
    acc = v[starts]
    for j in range(1, int(lens.max())):
        sel = (lens > j).nonzero().squeeze(1)
        acc[sel] += v[starts[sel] + j]
    return acc


def _device_csr(ctx, nt, nc, parts, to_host):
    """A sparse count matrix on the device as canonical CSR: (row pointers int64 [nt + 1], cell indices int32
    ascending and unique per gene, counts int32 / int64, (min, max, total) of the stored counts).  The counts are
    what ``toarray()`` followed by the dense path's cast to an integer type gives: duplicates summed in the value
    dtype, then floats truncated.  O(nnz) work; the caller's arrays are not modified."""
    fmt, a, b, v = parts
    if to_host:
        if np.dtype(v.dtype).kind not in 'biuf':
            v = np.asarray(v).astype(np.float64)
        kind, bits = np.dtype(v.dtype).kind, 8 * np.dtype(v.dtype).itemsize
        a, b, v = _ship(ctx, a), _ship(ctx, b), _ship(ctx, v)
    else:
        kind = 'b' if v.dtype == torch.bool else 'f' if v.dtype.is_floating_point else 'i' if v.dtype.is_signed else 'u'
        bits = 8 * v.element_size()
        if v.dtype == torch.bool:
            v = v.view(torch.uint8)
    dev = ctx.device
    nnz = v.numel()
    if nc > np.iinfo(np.int32).max:
        raise ValueError('sparse reads: at most %d cells.' % np.iinfo(np.int32).max)
    canonical = False
    if fmt == 'csr':
        indptr = a.to(torch.int64)
        canonical = nnz <= 1
        if not canonical:
            inc = b[1:] > b[:-1]                                # cell indices ascending within a gene ...
            first = indptr[1:-1]
            first = first[(first > 0) & (first < nnz)]
            inc[first - 1] = True                               # ... and anything across a gene boundary
            canonical = bool(inc.all())
            del inc, first
    summed = False
    if canonical:
        col = b.to(torch.int32)
    else:
        # (gene, cell) keys in storage order -> stable sort -> duplicates summed in storage order
        if fmt == 'csr':
            row, col = torch.repeat_interleave(torch.arange(nt, device=dev), torch.diff(indptr), output_size=nnz), b.long()
        elif fmt == 'csc':
            row = b.long()
            col = torch.repeat_interleave(torch.arange(nc, device=dev), torch.diff(a.to(torch.int64)), output_size=nnz)
        else:
            row, col = a.long(), b.long()
        key = row * nc + col
        del row, col
        if nnz > 1 and not bool((key[1:] > key[:-1]).all()):
            key, perm = torch.sort(key, stable=True)
            v = v[perm]
            del perm
            first = torch.ones(nnz, dtype=torch.bool, device=dev)
            first[1:] = key[1:] != key[:-1]
            starts = first.nonzero().squeeze(1)
            del first
            if starts.numel() < nnz:
                v = _sum_runs(v.to(torch.int64) if kind != 'f' else v, starts, nnz)
                key = key[starts]
                summed = True
            del starts
        indptr = torch.zeros(nt + 1, dtype=torch.int64, device=dev)
        torch.cumsum(torch.bincount(key // nc, minlength=nt), 0, out=indptr[1:])
        col = (key % nc).to(torch.int32)
        del key
    # the dense path's integer counts: floats truncated, integer sums wrapped to the value dtype's width
    if kind == 'f':
        if nnz and bool((~(v.abs() < 2.0 ** 63)).any()):
            raise ValueError('Negative value in d detected.')          # NaN / inf cast to the most negative int64
        v = v.to(torch.int64)
    elif kind == 'b':
        v = (v != 0).to(torch.int32)
    elif kind == 'u' and bits < 64:
        v = v.to(torch.int64) & ((1 << bits) - 1)
    elif kind == 'i' and bits < 64 and summed:
        v = ((v + (1 << (bits - 1))) & ((1 << bits) - 1)) - (1 << (bits - 1))
    elif v.dtype not in (torch.int32, torch.int64):
        v = v.to(torch.int64)
    nnz = v.numel()                                             # after duplicates were summed
    stats = (0, 0, 0)
    if nnz:
        scan = torch.empty(3, dtype=torch.int64, device=dev)
        _lib.check(ctx.lib.nsr_lcpm_scan(ctx.handle, engine._stream(), v.data_ptr(), v.element_size(), 1, nnz, nnz,
                                         scan.data_ptr()), "nsr_lcpm_scan")
        engine.LAUNCHES += 1
        stats = tuple(int(x) for x in scan.cpu().tolist())
    if v.dtype == torch.int64 and stats[0] >= -2 ** 31 and stats[1] < 2 ** 31:
        v = v.to(torch.int32)                                   # a 64 KB tile per CTA instead of 128 KB
    if nnz == 0:                                                # the kernels take non-null arrays
        col, v = torch.zeros(1, dtype=torch.int32, device=dev), torch.zeros(1, dtype=torch.int32, device=dev)
    return indptr.contiguous(), col.contiguous(), v.contiguous(), stats


def lcpm(reads, normalize=True, nth=0, ntot=None, varscale=0, seed=None, lowmem=True, nocov=False, device=None,
         noise=None):
    """Computes Bayesian log CPM from raw read counts: ``(lcpm, mean|None, var|None, cov|None)``
    with the reference's shapes (lcpm.py:29-66).  ``reads``: a (genes x cells) count matrix - numpy / CUDA strided,
    or sparse (scipy.sparse on the host, torch sparse CSR / CSC / COO on the device; see the module docstring),
    with the dense result on the same side.  ``nth`` is accepted and ignored."""
    if reads.ndim != 2:
        raise ValueError('reads must have 2 dimensions.')
    if varscale < 0:
        raise ValueError('varscale must be non-negative.')
    if not normalize or ntot is not None or varscale != 0:
        logging.warning("Modifying keyword arguments other than nth or seed is neither recommended nor supported "
                        "for function 'lcpm'. Do so at your own risk.")
    to_host = not _is_dev(reads)
    ctx = engine.context(device if device is not None else (reads.device if not to_host else None))
    dev = ctx.device
    parts = _sparse_parts(reads)
    csr = None
    if to_host and seed is not None:
        np.random.seed(seed)                                # lcpm.py:86-87
    if parts is not None:
        nt, nc = reads.shape
        itemsize = 0
    elif to_host:
        r = np.ascontiguousarray(reads)
        if not np.issubdtype(r.dtype, np.integer):
            r = r.astype(np.int64)                          # lcpm.py:129, 147
        if r.dtype not in (np.int32, np.int64):
            r = r.astype(np.int64 if r.dtype.itemsize > 4 or r.dtype.kind == 'u' and r.dtype.itemsize == 4 else np.int32)
        src = torch.from_numpy(r)
    else:
        src = reads
        if src.dtype not in (torch.int32, torch.int64):
            src = src.to(torch.int64)
        if src.stride(1) != 1:
            src = src.contiguous()
    if parts is None:
        nt, nc = src.shape
        itemsize = src.element_size()
    resample = varscale != 0
    with torch.cuda.device(dev):
        step = max(1, min(nt, min(_ROW_CHUNK_BYTES, hoststage.STAGE_BYTES) // max(1, 8 * nc))) if to_host else nt
        blocks = [(g0, min(nt, g0 + step)) for g0 in range(0, nt, step)]
        single = len(blocks) == 1
        held = {}
        if parts is not None:
            # sparse counts: canonical CSR on the device for both passes, O(nnz) (never genes x cells)
            csr = _device_csr(ctx, nt, nc, parts, to_host)
            itemsize = csr[2].element_size()
            src = None
        # both passes read the counts: a host matrix that fits comfortably stays on the device in between
        keep_on_device = to_host and nt * nc * itemsize <= _HOLD_BYTES
        n_out = 1 + (0 if lowmem else 2)
        stage = hoststage.RowBlocks(ctx, src, step, out_row_bytes=8 * nc * n_out, tag="lcpm") if to_host else None

        # one launch of a pass on row block i: the CSR kernels, or the strided ones on blk (rows of the dense counts)
        def colstats(i, blk, lut, lut_exp, sd_p, nz_p, ldn, sd_key, part, minmax):
            g0, g1 = blocks[i]
            if csr is not None:
                indptr, idx, val, _ = csr
                _lib.check(ctx.lib.nsr_lcpm_colstats_csr(ctx.handle, engine._stream(), indptr[g0:].data_ptr(),
                                                         idx.data_ptr(), val.data_ptr(), itemsize, g1 - g0, nc,
                                                         lut.data_ptr(), lut_exp.data_ptr() if lut_exp is not None else None,
                                                         lut.numel(), sd_p, nz_p, ldn, sd_key, g0, part.data_ptr(),
                                                         minmax.data_ptr()),
                           "nsr_lcpm_colstats_csr")
            else:
                _lib.check(ctx.lib.nsr_lcpm_colstats(ctx.handle, engine._stream(), blk.data_ptr(), itemsize, g1 - g0, nc,
                                                     blk.stride(0) if g1 - g0 > 1 else nc, lut.data_ptr(),
                                                     lut_exp.data_ptr() if lut_exp is not None else None,
                                                     lut.numel(), sd_p, nz_p, ldn, sd_key, g0, part.data_ptr(),
                                                     minmax.data_ptr()),
                           "nsr_lcpm_colstats")
            engine.LAUNCHES += 2

        def apply(i, blk, lut, sd_p, nz_p, ldn, sd_key, shift, res):
            g0, g1 = blocks[i]
            if csr is not None:
                indptr, idx, val, _ = csr
                _lib.check(ctx.lib.nsr_lcpm_apply_csr(ctx.handle, engine._stream(), indptr[g0:].data_ptr(), idx.data_ptr(),
                                                      val.data_ptr(), itemsize, g1 - g0, nc, lut.data_ptr(), lut.numel(),
                                                      sd_p, nz_p, ldn, sd_key, g0,
                                                      shift.data_ptr() if shift is not None else None, res.data_ptr(), nc),
                           "nsr_lcpm_apply_csr")
            else:
                _lib.check(ctx.lib.nsr_lcpm_apply(ctx.handle, engine._stream(), blk.data_ptr(), itemsize, g1 - g0, nc,
                                                  blk.stride(0) if g1 - g0 > 1 else nc, lut.data_ptr(), lut.numel(), sd_p,
                                                  nz_p, ldn, sd_key, g0, shift.data_ptr() if shift is not None else None,
                                                  res.data_ptr(), nc),
                           "nsr_lcpm_apply")
            engine.LAUNCHES += 1

        def block(i):
            g0, g1 = blocks[i]
            if i in held:
                return held[i]
            blk = stage.fetch(g0, g1) if to_host else src[g0:g1]
            if single or keep_on_device:
                held[i] = blk
            return blk

        i64 = torch.iinfo(torch.int64)
        minmax = torch.tensor([i64.max, i64.min], dtype=torch.int64, device=dev)
        lut_var = lut_sd = None
        noise_d = None
        key = 0
        if resample:
            # the standard-deviation table must cover every count and needs the total: one extra read
            # (pass 0: min / max / total)
            scan = torch.empty(3, dtype=torch.int64, device=dev)
            acc = None
            if csr is not None:                             # the stored counts, and 0 if some entry is not stored
                mn, mx, tot = csr[3]
                implicit = int(csr[0][-1]) < nt * nc
                acc = np.array([min(mn, 0) if implicit else mn, max(mx, 0) if implicit else mx, tot])
            for i, (g0, g1) in enumerate(blocks if csr is None else ()):
                blk = block(i)
                _lib.check(ctx.lib.nsr_lcpm_scan(ctx.handle, engine._stream(), blk.data_ptr(), itemsize, g1 - g0, nc,
                                                 blk.stride(0) if g1 - g0 > 1 else nc, scan.data_ptr()), "nsr_lcpm_scan")
                engine.LAUNCHES += 1
                cur = scan.cpu().numpy().copy() if nt and nc else np.array([0, 0, 0])
                acc = cur if acc is None else np.array([min(acc[0], cur[0]), max(acc[1], cur[1]), acc[2] + cur[2]])
            if acc is None:
                acc = np.array([0, 0, 0])
            if acc[0] < 0:
                raise ValueError('Negative value in d detected.')                # lcpm.py:88-89
            t0 = (int(acc[2]) if ntot is None else int(ntot)) + 2
            assert t0 > 2
            counts1 = torch.arange(1, int(acc[1]) + 2, dtype=torch.float64, device=dev)
            lut = torch.special.digamma(counts1).contiguous()                                    # :96-103 (+ const)
            lut_exp = None
            t0_t = torch.tensor(float(t0), dtype=torch.float64, device=dev)
            lut_var = (_trigamma(counts1) - _trigamma(t0_t)).contiguous()                        # :104-109
            lut_sd = torch.sqrt(lut_var * float(varscale)).contiguous()                          # :148-150
            if noise is None and to_host:
                noise = np.random.randn(nt, nc)             # the reference's own stream (:150)
            if noise is not None:
                noise_d = noise if isinstance(noise, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(noise, dtype=np.float64))
                if tuple(noise_d.shape) != (nt, nc):
                    raise ValueError('noise must have the shape of reads.')
            else:
                key = int(seed) if seed is not None else int(torch.randint(0, 2 ** 62, (1,)).item())
        else:
            # digamma(1 + c) and its exponential for the counts a table serves (larger ones are evaluated in
            # the kernels): independent of the data, built once per device
            lut, lut_exp = _tables(dev)

        def noise_args(g0, g1):
            if not resample:
                return None, None, 0, 0
            if noise_d is None:
                return lut_sd.data_ptr(), None, 0, key
            nb = noise_d[g0:g1].to(dev, torch.float64, non_blocking=True)
            if nb.stride(1) != 1:
                nb = nb.contiguous()
            keep.append(nb)
            return lut_sd.data_ptr(), nb.data_ptr(), nb.stride(0) if g1 - g0 > 1 else nc, 0

        keep = []
        # pass 1: per-cell statistics (+ smallest negative / largest count)
        col = torch.zeros((3, nc), dtype=torch.float64, device=dev)
        for i, (g0, g1) in enumerate(blocks):
            blk = block(i) if csr is None else None
            part = torch.empty((3, nc), dtype=torch.float64, device=dev)
            sd_p, nz_p, ldn, sd_key = noise_args(g0, g1)
            colstats(i, blk, lut, lut_exp, sd_p, nz_p, ldn, sd_key, part, minmax)
            col += part
        # digamma(total + 2), the constant of the reference's table: on the device, no host round trip
        total_t = col[1].sum() if ntot is None else torch.tensor(float(ntot), dtype=torch.float64, device=dev)
        psi_t0 = torch.special.digamma(total_t + 2.0)
        shift = psi_t0.expand(nc)                            # value = lut[c] - shift
        if normalize:                                        # lcpm.py:155-157: the constant cancels
            shift = torch.log(col[0]) - float(np.log(1e6))
        shift = shift.contiguous()
        dcov = None
        if not nocov:                                        # lcpm.py:193-199
            t1 = torch.log(col[1])
            dcov = torch.stack([t1, nt - col[2], t1 ** 2])
        # one small device->host read for the checks the reference makes up front
        chk = torch.stack([minmax[0].to(torch.float64), total_t.to(torch.float64), (col[1] == 0).any().to(torch.float64),
                           torch.isfinite(shift).all().to(torch.float64)]).cpu().numpy()
        if chk[0] < 0:
            raise ValueError('Negative value in d detected.')                    # lcpm.py:88-89
        assert chk[1] + 2 > 2                                                    # :91
        if not nocov and chk[2]:
            raise ValueError('Found cell with no read at all. Please remove.')   # :195-196
        if not chk[3]:
            raise AssertionError('non-finite logCPM')                            # :201
        # pass 2: gather (+ resampling) + per-cell shift
        host_out = to_host
        out = torch.empty((nt, nc), dtype=torch.float64, device=dev) if not host_out else torch.empty((nt, nc), dtype=torch.float64)
        dmean = dvar = None
        if not lowmem:                                       # lcpm.py:160-190
            dmean = torch.empty_like(out)
            dvar = torch.zeros_like(out)
        lut_vs = None
        if not lowmem and resample and csr is not None:
            lut_vs = (lut_var * float(varscale)).contiguous()  # var = lut_var[c] * varscale, gathered by the apply pass
        for i, (g0, g1) in enumerate(blocks):
            blk = block(i) if csr is None else None
            res = out[g0:g1] if not host_out else torch.empty((g1 - g0, nc), dtype=torch.float64, device=dev)
            sd_p, nz_p, ldn, sd_key = noise_args(g0, g1)
            apply(i, blk, lut, sd_p, nz_p, ldn, sd_key, shift, res)
            if host_out:
                stage.store(out[g0:g1], res)
            if not lowmem:
                if resample:
                    m = torch.empty((g1 - g0, nc), dtype=torch.float64, device=dev)
                    apply(i, blk, lut, None, None, 0, 0, shift, m)
                    if csr is not None:
                        v = torch.empty((g1 - g0, nc), dtype=torch.float64, device=dev)
                        apply(i, None, lut_vs, None, None, 0, 0, None, v)
                    else:
                        v = lut_var[blk.long().clamp_(0, lut_var.numel() - 1)] * float(varscale)
                else:
                    m, v = res, None
                if host_out:
                    stage.store(dmean[g0:g1], m)
                    if v is not None:
                        stage.store(dvar[g0:g1], v)
                else:
                    dmean[g0:g1] = m
                    if v is not None:
                        dvar[g0:g1] = v
        if to_host:
            stage.close()
            torch.cuda.current_stream().synchronize()
            return (out.numpy(), None if dmean is None else dmean.numpy(), None if dvar is None else dvar.numpy(),
                    None if dcov is None else dcov.cpu().numpy())
        return (out, dmean, dvar, dcov)
