"""``normalisr.coex.coex`` on the GPU (reference src/normalisr/coex.py:4-48), and two extensions:
``coexnet``, the reference's ``coex`` -> ``binnet`` pipeline as one call, and ``coextop``, every gene's k
strongest partners without a genes x genes matrix."""
import numpy as np
import torch

# Device bytes of the two strip buffers (P and dot) of coextop; the strip is the largest multiple of 128 rows
# that fits, and at least 128 rows.
_STRIP_BYTES = 1 << 30


def coex(dt, dc, **ka):
    """Co-expression for all gene pairs: ``(P, dot, var)``.

    dt: (n_gene, n_cell) normalised expression; dc: (n_cov, n_cell) covariates.
    P and dot are (n_gene, n_gene) with a zero diagonal, var is (n_gene,);
    Pearson R = dot / sqrt(var_i var_j)  (coex.py:30-34).
    Keyword arguments as the reference (``nth``, ``bsx``, ``bsy``, ``dimreduce`` ...; the
    batch-size / thread ones are accepted and ignored)."""
    from .association import association_tests
    ka.pop('bs', None)      # documented at coex.py:38; the reference itself rejects it downstream
    ans = association_tests(dt, None, dc, **ka)
    return (ans[0], ans[1], ans[4])


def coexnet(dt, dc, qcut, sparse=False, edge_values=False, devices=None, device=None, precision='default',
            dimreduce=0):
    """Co-expression network straight from the expression matrix: ``binnet(coex(dt, dc)[0], qcut)`` without
    P or dot ever leaving the GPUs.  Returns ``(net, var)``, or ``(net, var, P_e, dot_e)`` with ``edge_values``.

    net: the binary network, exactly ``binnet(coex(dt, dc)[0], qcut, sparse=sparse)`` - dense bool (G, G), or
    with ``sparse=True`` CSR with bool data (scipy for host input, torch sparse CSR for CUDA input); var: coex's
    var.  ``edge_values`` (``sparse=True`` only): P and dot at the edges, float64 arrays aligned with
    ``net.indices``, bit-identical to coex's P and dot there.

    One GPU (``device``, host or CUDA input): residualise and contract into P and dot on the device, then the
    binnet kernels on the device P; only the network (and the edge values) goes to the host.
    ``devices`` with more than one GPU (host input): ``parallel.coexnet_all_devices``.  ``precision`` and
    ``dimreduce`` as for ``coex``.  Raises like ``coex`` and ``binnet``."""
    from . import engine, parallel
    from ._lib import MODE_COEX
    from .association import _is_dev, _residualize_any, basis_and_dof
    from .binnet import device_net
    if len(dt.shape) != 2 or len(dc.shape) != 2:
        raise ValueError('Incorrect dx/dy/dc size.')
    n_gene, n = dt.shape
    if dc.shape[1] != n:
        raise ValueError('Unmatching dx/dy/dc dimensions.')
    if n_gene <= 1:
        raise ValueError('Wrong shape of net or namet.')
    if qcut <= 0 or qcut >= 1:
        raise ValueError('Q-value cutoff must be between 0 and 1.')
    if edge_values and not sparse:
        raise ValueError('edge_values needs sparse=True (values aligned with net.indices).')
    if precision not in engine.PRESETS:
        raise ValueError('Unknown precision {}'.format(precision))
    if np.ndim(dimreduce) != 0:
        raise ValueError('dimreduce must be a scalar.')
    dimreduce = int(dimreduce)
    if devices is not None:
        devs = parallel.visible_devices(devices)
        if len(devs) > 1:
            if _is_dev(dt) or device is not None:
                raise ValueError('devices= takes host inputs (the matrices are spread over the GPUs).')
            return parallel.coexnet_all_devices(dt, dc, qcut, sparse=sparse, edge_values=edge_values, devices=devs,
                                                precision=precision, dimreduce=dimreduce)
        device = devs[0]
    to_host = not _is_dev(dt)
    ctx = engine.context(device if device is not None else (dt.device if not to_host else None))
    n_slices, n_products = engine.PRESETS[precision]
    Qt_dev, _, _, dof_a = basis_and_dof(ctx, dc, n, dimreduce)
    with torch.cuda.device(ctx.device):
        A = _residualize_any(ctx, dt, Qt_dev, n_slices, False)
        P = torch.empty((n_gene, n_gene), dtype=torch.float64, device=ctx.device)
        D = torch.empty_like(P)
        engine.contract(ctx, MODE_COEX, A, A, engine.coex_tiles(n_gene), dof_a, P, D, n_products)
        res = device_net(ctx, P, qcut, sparse, to_host, D=D if edge_values else None)
        var = A.var.cpu().numpy() if to_host else A.var
        if edge_values:
            return res[0], var, res[1], res[2]
        return res, var


def coextop(dt, dc, k, device=None, precision='default', dimreduce=0, devices=None):
    """Every gene's k strongest co-expression partners: ``(idx, P_k, dot_k, var)``.

    idx: (G, k) int64; row i holds the k columns j != i with the largest r2_ij = dot_ij^2 / (var_i var_j),
    in descending order, ties to the smaller column.  P_k, dot_k: (G, k) float64, coex's P and dot at
    those entries (bit for bit); var: coex's var.  r2 ranks pairs like P wherever P has not underflowed
    (the degrees of freedom are common to all pairs), and unlike P it still ranks them at atlas sizes.

    The genes x genes matrices never exist: the upper triangle is contracted one strip of 128-row tiles at a
    time into two strip buffers of at most ``_STRIP_BYTES``, and after each strip one kernel folds the strip's
    pairs into every row's running top k (32 B per slot, G k slots).  One GPU (``device``); numpy in -> numpy
    out, CUDA tensors in -> CUDA tensors out.  ``devices`` with more than one GPU (host input, numpy out):
    ``parallel.coextop_all_devices``, the strips dealt out to the GPUs and the partial lists merged on the
    devices, bit-identical to one GPU; a list of one device runs the one-GPU path there.
    1 <= k <= min(G - 1, 2048).  ``precision`` and ``dimreduce`` as for ``coex``."""
    from . import engine, parallel
    from ._lib import TILE, TOPK_MAX
    from .association import _is_dev, _outs, _residualize_any, basis_and_dof
    if len(dt.shape) != 2 or len(dc.shape) != 2:
        raise ValueError('Incorrect dx/dy/dc size.')
    n_gene, n = dt.shape
    if dc.shape[1] != n:
        raise ValueError('Unmatching dx/dy/dc dimensions.')
    if n_gene <= 1:
        raise ValueError('Wrong shape of net or namet.')
    if np.ndim(k) != 0 or int(k) != k or not 1 <= int(k) <= min(n_gene - 1, TOPK_MAX):
        raise ValueError('k must be an integer in [1, min(n_gene - 1, {})].'.format(TOPK_MAX))
    k = int(k)
    if precision not in engine.PRESETS:
        raise ValueError('Unknown precision {}'.format(precision))
    if np.ndim(dimreduce) != 0:
        raise ValueError('dimreduce must be a scalar.')
    dimreduce = int(dimreduce)
    if devices is not None:
        devs = parallel.visible_devices(devices)
        if len(devs) > 1:
            if _is_dev(dt) or device is not None:
                raise ValueError('devices= takes host inputs (the matrices are spread over the GPUs).')
            return parallel.coextop_all_devices(dt, dc, k, devices=devs, precision=precision, dimreduce=dimreduce)
        device = devs[0]
    to_host = not _is_dev(dt)
    ctx = engine.context(device if device is not None else (dt.device if not to_host else None))
    n_slices, n_products = engine.PRESETS[precision]
    Qt_dev, _, _, dof_a = basis_and_dof(ctx, dc, n, dimreduce)
    with torch.cuda.device(ctx.device):
        A = _residualize_any(ctx, dt, Qt_dev, n_slices, False)
        k_chunk = engine.plan_k_chunk(A, A, n_products)
        state = torch.empty((n_gene, k, 4), dtype=torch.float64, device=ctx.device)
        top_strips(ctx, A, dof_a, n_products, k_chunk, state, 0, (n_gene + TILE - 1) // TILE)
        res = engine.topk_finish(ctx, state) + (A.var,)
        if to_host:
            res = _outs(res)
    return res


def top_strips(ctx, A, dof_a, n_products, k_chunk, state, a, b):
    """coextop's selection over the strips of tile rows [a, b): each strip of at most ``_STRIP_BYTES`` is
    contracted (upper triangle, columns from the strip's first row to G) and folded into ``state`` ((G, k, 4)
    slots).  The range (0, n_tiles) is the whole selection and initialises the state; any other range needs a
    state set empty by ``engine.topk_reset`` first and leaves the top k of its own pairs (``nsr_topk_merge``
    then combines the ranges)."""
    from . import engine
    from ._lib import MODE_COEX_UPPER, TILE
    n_gene, k = state.shape[0], state.shape[1]
    n_tiles = (n_gene + TILE - 1) // TILE
    strip = max(1, _STRIP_BYTES // (16 * TILE * n_gene))
    if b <= a:
        return
    rows = min(min(strip, b - a) * TILE, n_gene)
    Ps = torch.empty((rows, n_gene), dtype=torch.float64, device=ctx.device)
    Ds = torch.empty_like(Ps)
    for a0 in range(a, b, strip):
        b0 = min(a0 + strip, b)
        r0, r1 = a0 * TILE, min(b0 * TILE, n_gene)
        engine.contract(ctx, MODE_COEX_UPPER, A, A, engine.upper_tiles(a0, b0, a0, n_tiles), dof_a, Ps, Ds,
                        n_products, k_chunk=k_chunk, row0=r0)
        engine.topk_strip(ctx, Ps, Ds, r0, r1, A.var, k, state)
