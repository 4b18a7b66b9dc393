"""``normalisr.coex.coex`` on the GPU (reference src/normalisr/coex.py:4-48), and ``coexnet``, the
reference's ``coex`` -> ``binnet`` pipeline as one call (an extension)."""
import numpy as np
import torch


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
