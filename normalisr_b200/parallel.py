"""Multi-GPU co-expression / DE: one process per GPU, torch.distributed (NCCL) for the single
exchange step.  Replaces the reference's thread pool over tiles (``parallel.autopooler``,
parallel.py:12-74, used at association.py:997).

The path shards naturally (SURVEY.md 8e):
  * every rank residualises and quantises its own block of genes (covariates are tiny and
    replicated); blocks are equal multiples of the 128-row tile;
  * the int8 digit planes (+ per-row quantum and variance) are exchanged ONCE.  Default schedule
    ("pairs"): the unordered block pairs {i, j} are dealt out on a circulant - rank r computes its
    diagonal block and the pairs (r, r+d mod W) for d = 1 .. W/2 (for even W the pairs at distance
    W/2 are split in two halves between their two owners).  Every rank therefore
    needs only W/2 remote blocks instead of W-1, receives them in W/2 point-to-point rounds in
    which all ranks send and receive at once, and contracts block pair d while round d+1 is in
    flight.  The older schedule ("allgather": one all-gather, then a strip of tile rows per rank)
    is kept for comparison;
  * no further communication: rank r ends with the rows of its block of P / dot for the column
    blocks it owns; ``gather_dense`` mirrors them into the full symmetric matrices;
  * one result for one caller (``home``): every GPU also writes the transposes of what it computes and copies
    its rectangles straight into ONE (n_gene, n_gene) host P and dot - under torchrun a page-locked mapping
    shared by the ranks (``coex_host`` + ``shared_host_matrices``), from one process the caller's own arrays
    (``coex_all_devices``, one worker thread per GPU; ``de_all_devices`` for de);
  * host inputs: the diagonal block of a rank is contracted in strips while its rows are still arriving
    (``diag_block_streamed``), and block pairs leave for the host in column strips with their own completion
    counters (``pair_strips``), so copy-in, tensor work and copy-out overlap.
Because the sums over cells are exact integers, every schedule gives bit-identical results.
"""
import collections
import logging

import numpy as np
import torch
import torch.distributed as dist

from . import engine
from ._lib import MAX_SEGMENTS, MODE_COEX_RECT, MODE_COEX_UPPER, MODE_DE, TILE, TOPK_MAX_PARTS
from .association import basis_and_dof, covariate_basis_device


def row_split(rows, world):
    """Contiguous, equally sized row blocks (last one short or empty): block size, a multiple of
    the tile so that no output tile straddles two blocks."""
    t = (rows + TILE - 1) // TILE
    return ((t + world - 1) // world) * TILE


def block_rows(rows, world, k):
    """Number of valid rows in block k."""
    blk = row_split(rows, world)
    return int(min(max(rows - k * blk, 0), blk))


def exchange_plan(world, rank):
    """Rounds of the block exchange for ``rank``: [(send_to, recv_from, parity)], round d-1 brings
    block (rank + d) mod world.  parity is None for a pair this rank computes in full, or 0 / 1 when
    the pair is shared with its other owner (even world, distance world/2): this rank takes the tiles
    ``pair_tiles`` selects for that parity (one half of the block pair, cut along block lo)."""
    plan = []
    for d in range(1, world // 2 + 1):
        src = (rank + d) % world
        parity = None
        if world % 2 == 0 and d == world // 2:
            parity = 0 if rank < src else 1
        plan.append(((rank - d) % world, src, parity))
    return plan


def pair_tiles(rows_a, rows_b, parity=None):
    """Tiles of the (rows_a x rows_b) block pair this rank computes.  A shared pair {lo, hi} (parity set)
    is cut along the tile rows of block lo: the lower-numbered owner (parity 0, its A = block lo) takes
    the first half of them, the other owner (parity 1, its B = block lo) the rest - two rectangles, so
    each owner's share is one rectangular block of the output (a 2-D copy home, no tile masks)."""
    tl = engine.rect_tiles(rows_a, rows_b)
    if parity is not None and len(tl):
        if parity == 0:
            tl = tl[tl[:, 0] < shared_cut(rows_a)]
        else:
            tl = tl[tl[:, 1] >= shared_cut(rows_b)]
    return np.ascontiguousarray(tl, dtype=np.int32).reshape(-1, 2)


def pair_strips(tl, rect, n_sub):
    """Cut the tiles ``tl`` of one block pair (covering rows x columns ``rect`` = (a0, a1, b0, b1) of the pair) into
    at most ``n_sub`` strips of whole tile columns: [(tiles, (a0, a1, c_lo, c_hi))], the tiles of every strip in
    their original order, the strips' column ranges a partition of [b0, b1).  One strip = the input."""
    a0, a1, b0, b1 = rect
    cols = np.unique(tl[:, 1]) if len(tl) else np.zeros(0, np.int32)
    if n_sub <= 1 or len(cols) <= 1:
        return [(np.ascontiguousarray(tl, dtype=np.int32).reshape(-1, 2), rect)]
    out = []
    for part in np.array_split(cols, min(n_sub, len(cols))):
        sel = tl[(tl[:, 1] >= part[0]) & (tl[:, 1] <= part[-1])]
        out.append((np.ascontiguousarray(sel, dtype=np.int32).reshape(-1, 2),
                    (a0, a1, max(b0, int(part[0]) * TILE), min(b1, (int(part[-1]) + 1) * TILE))))
    return out


def shared_cut(rows_lo):
    """Tile row of block lo at which a shared block pair is cut between its two owners."""
    return ((rows_lo + TILE - 1) // TILE + 1) // 2


def owned_tile_mask(n_gene, world, rank):
    """Boolean (tile rows of block ``rank``, all tile columns): which output tiles the pairs
    schedule computes on ``rank`` (diagonal block: upper triangle including diagonal tiles)."""
    blk = row_split(n_gene, world)
    tb = blk // TILE
    t = (n_gene + TILE - 1) // TILE
    ta = (block_rows(n_gene, world, rank) + TILE - 1) // TILE
    m = np.zeros((ta, t), dtype=bool)
    for i in range(ta):
        m[i, rank * tb + i: rank * tb + ta] = True
    for _, src, parity in exchange_plan(world, rank):
        for ti, tj in pair_tiles(block_rows(n_gene, world, rank), block_rows(n_gene, world, src), parity):
            m[ti, src * tb + tj] = True
    return m


def start_exchange(local, group=None):
    """Post every round of the block exchange (non-blocking).  Returns [(src, parity, Sliced, works)]
    in round order; ``wait_block`` makes the current stream wait for one round."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)

    def peer(r):
        return dist.get_global_rank(group, r) if group is not None else r

    rounds = []
    for dst, src, parity in exchange_plan(world, rank):
        buf = engine.Sliced(local.rows_alloc, local.n, local.n_slices, local.slices.device)
        ops = []
        for t_send, t_recv in ((local.slices, buf.slices), (local.quantum, buf.quantum), (local.var, buf.var)):
            ops.append(dist.P2POp(dist.isend, t_send, peer(dst), group))
            ops.append(dist.P2POp(dist.irecv, t_recv, peer(src), group))
        rounds.append((src, parity, buf, dist.batch_isend_irecv(ops)))
    return rounds


def wait_block(works):
    for w in works:
        w.wait()


def strip_bounds(n_tile_rows, world):
    """Tile-row strips [a_k, b_k) with (nearly) equal numbers of upper-triangular tiles.
    Tile row i holds n_tile_rows - i tiles."""
    total = n_tile_rows * (n_tile_rows + 1) // 2
    bounds = [0]
    acc, k = 0, 1
    for i in range(n_tile_rows):
        acc += n_tile_rows - i
        while k < world and acc >= total * k / world:
            bounds.append(i + 1)
            k += 1
    while len(bounds) < world:
        bounds.append(n_tile_rows)
    bounds.append(n_tile_rows)
    return [(bounds[k], max(bounds[k], bounds[k + 1])) for k in range(world)]


def strip_tiles(n_tile_rows, a, b, strip=12):
    """Upper-triangular tiles with tile row in [a, b), column-strip ordered for L2 reuse."""
    return engine.upper_tiles(a, b, a, n_tile_rows, strip)


def gather_sliced(local, rows_total, group=None):
    """All-gather equally sized row blocks of digit planes into one Sliced of rows_total rows."""
    world = dist.get_world_size(group)
    blk = local.rows_alloc
    full = engine.Sliced(blk * world, local.n, local.n_slices, local.slices.device)
    for s in range(local.n_slices):
        dist.all_gather_into_tensor(full.slices[s], local.slices[s].contiguous(), group=group)
    dist.all_gather_into_tensor(full.quantum, local.quantum, group=group)
    dist.all_gather_into_tensor(full.var, local.var, group=group)
    full.energy_max.copy_(local.energy_max)
    dist.all_reduce(full.energy_max, op=dist.ReduceOp.MAX, group=group)   # maxima over all ranks' rows
    full.rows = rows_total            # rows beyond rows_total are padding of the last block
    return full


_SYMM = {}            # (bytes, device, group) -> (symmetric uint8 buffer, handle) or None, decided once
# Plane exchange: "ce" = copy-engine pulls from peer-mapped memory (no SMs taken from the
# contraction; N = 2: 67.5 vs 72.9 ms per step), "nccl" = point-to-point send/recv kernels,
# "auto" = "ce" when peer-mapped (symmetric) memory can be set up on all ranks, else "nccl".
TRANSPORT = "auto"
PAIR_STRIPS = 8            # column strips per block pair when results go to the host (see contract_plan)
STREAM_DIAGONAL = True     # host inputs with one home matrix: the diagonal block is contracted while the block's rows arrive


def _symm_block(nbytes, device, group):
    """A buffer of ``nbytes`` every rank of ``group`` can map (torch symmetric memory over NVLink)."""
    key = (nbytes, torch.device(device).index, id(group))
    if key not in _SYMM:
        import torch.distributed._symmetric_memory as symm
        t = symm.empty(nbytes, dtype=torch.uint8, device=device)
        hdl = symm.rendezvous(t, group if group is not None else dist.group.WORLD)
        _SYMM[key] = (t, hdl)
    return _SYMM[key]


def _pull_rounds(ctx, local, rank, world, stores, pull):
    """Copy-engine variant of ``start_exchange``: every remote block is PULLED with an asynchronous copy
    on a side stream, so the exchange uses no SMs while the contraction runs.  Each copy is followed by a
    stream-ordered flag write (``nsr_stream_signal``): the persistent contraction launch, already running,
    starts on a block's tiles when its flag appears.  Round d lands in ``stores[d]`` (uint8, the size of
    ``Sliced.storage_bytes``); ``pull(src, store)`` queues on the current stream (the side stream) whatever
    the copy must wait for and the copy of block src into ``store``.  Returns [(src, parity, Sliced,
    [_FlagWork])]."""
    dev = local.slices.device
    side = _side_stream(dev, "pull")
    side.wait_stream(torch.cuda.current_stream())
    sync = _sync_words(ctx)
    sync.epoch += 1
    rounds = []
    for d, (_, src, parity) in enumerate(exchange_plan(world, rank)):
        with torch.cuda.stream(side):
            pull(src, stores[d])
            ev = torch.cuda.Event()
            ev.record(side)
            work = _FlagWork(ev, sync.ready_ptr(d + 1), sync.epoch)
            engine.stream_signal(ctx, work.flag_ptr, work.value, stream=side)
        buf = engine.Sliced(local.rows_alloc, local.n, local.n_slices, dev, storage=stores[d], fresh=False)
        rounds.append((src, parity, buf, [work]))
    return rounds


_SIDE = {}


def _side_stream(device, role):
    """One stream per device and role: "pull" brings remote blocks in, "send" takes results out."""
    key = (torch.device(device).index, role)
    if key not in _SIDE:
        _SIDE[key] = torch.cuda.Stream(device=device)
    return _SIDE[key]


class _SyncWords:
    """Per-device uint32 words shared with the persistent contraction launch: ready flags (one per
    segment, set to the step's epoch by the copy stream) and done counters (monotonic)."""

    def __init__(self, device):
        self.words = torch.zeros(64, dtype=torch.int32, device=device)
        self.epoch = 0
        self.done_expected = [0] * 16

    def ready_ptr(self, seg):
        return self.words.data_ptr() + 4 * seg

    def done_ptr(self, seg):
        return self.words.data_ptr() + 4 * (32 + seg)


_SYNC = {}


def _sync_words(ctx):
    key = ctx.device.index
    if key not in _SYNC:
        _SYNC[key] = _SyncWords(ctx.device)
    return _SYNC[key]


class _FlagWork:
    """A block a copy engine is bringing in (``_pull_rounds``): ``wait()`` makes the current stream wait for
    the copy's event (like a c10d Work); the single-launch contraction instead waits inside the kernel for
    the device flag the copy stream sets to ``value``."""

    def __init__(self, ev, flag_ptr, value):
        self.ev, self.flag_ptr, self.value = ev, flag_ptr, value

    def wait(self):
        torch.cuda.current_stream().wait_event(self.ev)


def _own_block(blk, rows, n, n_slices, device, storage=None):
    """A rank's block of ``blk`` rows for its ``rows`` genes, before they are residualised into it: the
    padding rows past them are zero planes with quantum 1, var 1."""
    out = engine.Sliced(blk, n, n_slices, device, storage=storage)
    if rows < blk:
        out.slices[:, rows:].zero_()
        out.quantum[rows:] = 1.0
        out.var[rows:] = 1.0
    return out


def residualize_block(ctx, x_block, Qt_dev, n_slices, blk, storage=None):
    """Residualise this rank's rows into a block padded to ``blk`` rows (``_own_block``)."""
    out = _own_block(blk, x_block.shape[0], x_block.shape[1], n_slices, ctx.device, storage=storage)
    if x_block.shape[0]:
        engine.residualize(ctx, x_block, Qt_dev, n_slices, out=out, row_offset=0)
    return out


def _timed(events, fn):
    """Run fn(); with ``events`` a list, bracket it with CUDA events on the current stream."""
    if events is None:
        return fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    res = fn()
    e1.record()
    events.append((e0, e1))
    return res


def _coex_pairs(ctx, local, n_gene, dof_a, n_products, group, out, events=None, out_host=None, symm=None, home=None,
                skip_diag=False):
    """Pairs schedule under torchrun on an already residualised block: post the exchange (copy-engine pulls
    from the peers' symmetric memory ``symm`` = (store, handle), else NCCL) and contract everything this rank
    owns (``_pairs``).  Returns (P, dot, var_all).  ``events`` (a list) receives one CUDA event pair per
    contraction launch (bench bookkeeping); ``out_host``, ``home``, ``skip_diag`` as for ``contract_plan``."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    rounds = []
    if world > 1 and symm is None:
        rounds = start_exchange(local, group)
    elif world > 1:
        hdl = symm[1]
        nbytes = symm[0].numel()
        hdl.barrier(channel=1, timeout_ms=60000)            # every rank's planes are written
        side = _side_stream(local.slices.device, "pull")
        stores = []
        for _ in exchange_plan(world, rank):
            stores.append(torch.empty(nbytes, dtype=torch.uint8, device=local.slices.device))
            stores[-1].record_stream(side)
        rounds = _pull_rounds(ctx, local, rank, world, stores, lambda src, store: store.copy_(
            hdl.get_buffer(src, (nbytes,), torch.uint8, 0), non_blocking=True))
    P, D = _pairs(ctx, local, rounds, rank, world, n_gene, dof_a, n_products, out, events, out_host, home, skip_diag)
    var_all = local.var
    if world > 1:
        var_all = torch.empty(local.rows_alloc * world, dtype=torch.float64, device=local.var.device)
        dist.all_gather_into_tensor(var_all, local.var, group=group)
    return P, D, var_all[:n_gene]


def _pairs(ctx, local, rounds, rank, world, n_gene, dof_a, n_products, out, events=None, out_host=None, home=None,
           skip_diag=False, gather=None):
    """Everything ``rank`` owns under the pairs schedule, given its residualised block and the ``rounds`` of
    the exchange (``contract_plan``): one optimistic pass over the cells, then the int32 partial sums are
    bounded from the digit energies of this rank's rows and of every block it used (the energies of the
    remote blocks travel with them, so no collective is needed) and the plan is redone in cell chunks if the
    bound fails (not observed below ~260k cells).  Returns (P, dot)."""
    P, D = contract_plan(ctx, local, rounds, rank, world, n_gene, dof_a, n_products, 0, out, events, out_host,
                         home=home, skip_diag=skip_diag, gather=gather)
    for r in rounds:
        wait_block(r[3])
    em_a = local.energy_max.cpu().numpy()
    em_b = em_a
    for r in rounds:
        em_b = np.maximum(em_b, r[2].energy_max.cpu().numpy())     # NaN (non-finite input) propagates
    k_chunk = engine.plan_k_chunk(local, local, n_products, energies=(em_a, em_b))
    if k_chunk:
        P, D = contract_plan(ctx, local, [(r[0], r[1], r[2], []) for r in rounds], rank, world, n_gene, dof_a,
                             n_products, k_chunk, (P, D), None, out_host, home=home, gather=gather)
    return P, D


def _segment_rect(rows_a, rows_b, parity):
    """(a0, a1, b0, b1): the rows of A x rows of B that ``pair_tiles`` covers for this parity."""
    if parity == 0:
        return 0, min(shared_cut(rows_a) * TILE, rows_a), 0, rows_b
    if parity == 1:
        return 0, rows_a, min(shared_cut(rows_b) * TILE, rows_b), rows_b
    return 0, rows_a, 0, rows_b


_MIRROR = {}


def _mirror_pair(device, k, blk):
    """(P, dot) buffers (blk x blk) that receive the transposed copy of block pair k of this device; kept
    per device so that the device-to-host copies of one call never outlive their source."""
    key = (torch.device(device).index, k, blk)
    if key not in _MIRROR:
        _MIRROR[key] = (torch.empty((blk, blk), dtype=torch.float64, device=device),
                        torch.empty((blk, blk), dtype=torch.float64, device=device))
    return _MIRROR[key]


Segment = collections.namedtuple("Segment", "src rows_b col0 diagonal tiles rect k works")
Segment.__doc__ = """One segment of ``contract_plan``: the rows of block ``rank`` x block ``src`` (``rows_b`` rows, output
columns from ``col0``); ``diagonal`` for the rank's own block (upper-triangular tiles, mirrored into P itself);
``tiles`` (k, 2) int32 within the block pair; ``rect`` = (a0, a1, b0, b1) the rows x columns of the pair those
tiles cover; ``k`` the round (1-based) whose block is B and whose mirror buffer receives the transposes, 0 for
the diagonal; ``works`` what the block's arrival is waited for with ([] when it is there)."""


def plan_segments(rounds, rank, world, n_gene, k_chunk=0, single_launch=True, mirrored=False, skip_diag=False):
    """The segments ``contract_plan`` launches, on the host: the diagonal block (unless ``skip_diag``), then each
    non-empty block pair of ``rounds`` = [(src, parity, block, works)].  When the transposes are written
    (``mirrored``) and the launch is one flag-driven pass, a block pair is cut into column strips, each a segment
    of its own (same operands, its own ``done`` counter), so that a strip leaves while the next one is contracted
    instead of the whole rectangle waiting for its last tile."""
    blk = row_split(n_gene, world)
    rows_a = block_rows(n_gene, world, rank)
    if not rows_a:
        return []
    segs = []
    if not skip_diag:
        segs.append(Segment(rank, rows_a, rank * blk, True, engine.coex_tiles(rows_a), (0, rows_a, 0, rows_a), 0, []))
    pairs = [(k, src, parity, works) for k, (src, parity, _, works) in enumerate(rounds, 1)
             if block_rows(n_gene, world, src)]
    flag_driven = single_launch and not k_chunk and all(len(r[3]) == 0 or isinstance(r[3][0], _FlagWork) for r in rounds)
    for done, (k, src, parity, works) in enumerate(pairs):
        rows_b = block_rows(n_gene, world, src)
        tl = pair_tiles(rows_a, rows_b, parity)
        n_sub = 1
        if mirrored and len(tl) and flag_driven:
            n_sub = max(1, min(PAIR_STRIPS, (MAX_SEGMENTS - len(segs)) // (len(pairs) - done)))
        for sel, rect in pair_strips(tl, _segment_rect(rows_a, rows_b, parity), n_sub):
            segs.append(Segment(src, rows_b, src * blk, False, sel, rect, k, works))
    return segs


def contract_plan(ctx, local, rounds, rank, world, n_gene, dof_a, n_products, k_chunk, out=None, events=None,
                  out_host=None, single_launch=True, home=None, skip_diag=False, gather=None):
    """Contract everything ``rank`` owns under the pairs schedule: the upper triangle of its diagonal
    block, then the block pairs of ``rounds`` = [(src, parity, Sliced of block src, works)].
    ``works``: [] when the block is already there (the one-GPU emulation of the schedule in
    tests/test_gpu_parity.py), a ``_FlagWork`` when a copy engine is bringing it and will set a device
    flag (the kernel waits for it), anything else with ``wait()`` (NCCL) is waited for on the stream.
    One persistent launch over all segments (``plan_segments``, ``nsr_contract_segments``) unless a block
    arrives over NCCL - its kernels need SMs, which a waiting persistent launch would not release - or
    ``single_launch`` is off; then one launch per segment.  Returns (P, dot): rows of block ``rank`` x
    all n_gene columns, owned tiles filled in.

    Where the results go besides (P, dot), each segment as soon as its tiles are finished, on a
    side stream, while the launch continues:
      out_host = (P, dot) host tensors (rows of this rank, n_gene): the same layout as (P, dot);
      home     = (P, dot) host tensors (n_gene, n_gene), the FULL symmetric matrices of the reference
                 (association.py:1036-1057): the kernel also writes the transposed copy of everything it
                 computes (diagonal block: into P itself; block pair: into a (rows_b x rows_a) buffer) and
                 both rectangles are copied home, so that after all ranks are done every entry of both
                 triangles has been written exactly once.
      gather   = one (P, dot) pair of device tensors per rank (the (P, dot) of every rank's call, rows of its
                 block x n_gene, on that rank's GPU): as with ``home`` the kernel writes the transposed copies,
                 and those of block pair (rank, src) go peer to peer into gather[src] at the columns of this
                 block, so that every rank ends up holding COMPLETE rows of its block once all ranks are done.
    ``skip_diag``: the diagonal block is already done and on its way home (``diag_block_streamed``: contracted
    in strips while the block's rows were still arriving from the host); only the block pairs are launched."""
    blk = local.rows_alloc
    rows_a = block_rows(n_gene, world, rank)
    dev = local.slices.device
    if out is None:
        P = torch.zeros((max(rows_a, 1), n_gene), dtype=torch.float64, device=dev)
        D = torch.zeros_like(P)
    else:
        P, D = out
    local.rows = max(rows_a, 1)
    mirrored = home is not None or gather is not None
    segs = plan_segments(rounds, rank, world, n_gene, k_chunk, single_launch, mirrored, skip_diag)
    if not segs:
        return P, D
    r0 = rank * blk
    to_host = out_host is not None or mirrored            # (gather: to the peers)
    copy_stream = _side_stream(dev, "send") if to_host else None
    main = torch.cuda.current_stream()
    mbufs = {sg.k: _mirror_pair(dev, sg.k, blk) for sg in segs if mirrored and not sg.diagonal}

    def operands(sg):
        """segment sg as engine.contract_segments takes it"""
        B = local if sg.diagonal else rounds[sg.k - 1][2]
        B.rows = sg.rows_b
        op = dict(B=B, rows_b=sg.rows_b, col0=sg.col0, diagonal=sg.diagonal)
        if mirrored and sg.diagonal:
            op["mirror"] = (P.data_ptr() + 8 * r0, D.data_ptr() + 8 * r0, P.stride(0))
        elif mirrored:
            op["mirror"] = (mbufs[sg.k][0].data_ptr(), mbufs[sg.k][1].data_ptr(), blk)
        return op

    def send(sg):
        """queue the copies of segment sg's results on the copy stream"""
        c0 = sg.col0
        a0, a1, b0, b1 = sg.rect
        mbuf = mbufs.get(sg.k) if not sg.diagonal else None
        if out_host is not None:
            for src_t, dst_t in zip((P, D), out_host):
                engine.copy_rect_to_host(ctx, dst_t, 0, c0, src_t, 0, c0, rows_a, sg.rows_b, stream=copy_stream)
        if home is not None:
            for t, (src_t, dst_t) in enumerate(zip((P, D), home)):
                engine.copy_rect_to_host(ctx, dst_t, r0 + a0, c0 + b0, src_t, a0, c0 + b0, a1 - a0, b1 - b0,
                                         stream=copy_stream)
                if mbuf is not None:
                    engine.copy_rect_to_host(ctx, dst_t, c0 + b0, r0 + a0, mbuf[t], b0, a0, b1 - b0, a1 - a0,
                                             stream=copy_stream)
        if gather is not None and mbuf is not None:
            for t in range(2):
                engine.copy_rect_to_peer(ctx, gather[sg.src][t], b0, r0 + a0, mbuf[t], b0, a0, b1 - b0, a1 - a0,
                                         stream=copy_stream)

    flagged = all(len(sg.works) == 0 or isinstance(sg.works[0], _FlagWork) for sg in segs)
    if single_launch and flagged and len(segs) <= MAX_SEGMENTS:
        sync = _sync_words(ctx)
        track = to_host and not k_chunk
        ops = [operands(sg) for sg in segs]
        for i, (sg, op) in enumerate(zip(segs, ops)):
            if sg.works:
                op["ready"] = (sg.works[0].flag_ptr, sg.works[0].value)
            if track:
                op["done"] = sync.done_ptr(i)
        tl = np.concatenate([np.concatenate([np.full((len(sg.tiles), 1), i, np.int32), sg.tiles], axis=1)
                             for i, sg in enumerate(segs)])
        _timed(events, lambda: engine.contract_segments(ctx, local, ops, tl, dof_a, P, D, n_products, k_chunk=k_chunk))
        if to_host:
            if not track:
                copy_stream.wait_stream(main)
            for i, sg in enumerate(segs):
                if track:
                    # the epilogue counts every finished tile of the segment once per epilogue warp
                    sync.done_expected[i] += EPILOGUE_WARPS * len(sg.tiles)
                    engine.stream_wait_geq(ctx, sync.done_ptr(i), sync.done_expected[i], stream=copy_stream)
                send(sg)
            main.wait_stream(copy_stream)
        return P, D

    for sg in segs:
        wait_block(sg.works)
        tl = np.concatenate([np.zeros((len(sg.tiles), 1), np.int32), sg.tiles], axis=1)
        _timed(events, lambda: engine.contract_segments(ctx, local, [operands(sg)], tl, dof_a, P, D, n_products,
                                                        k_chunk=k_chunk))
        if to_host:
            copy_stream.wait_stream(main)
            send(sg)
    if copy_stream is not None:
        main.wait_stream(copy_stream)
    return P, D


EPILOGUE_WARPS = 8        # epilogue warps of the tcgen05 kernel (each counts a finished tile once)


def _coex_strip(ctx, local, n_gene, dof_a, n_products, group, out, events=None):
    """All-gather schedule: every rank gets all planes, then computes a strip of tile rows."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    full = gather_sliced(local, n_gene, group) if world > 1 else local
    full.rows = n_gene
    t = (n_gene + TILE - 1) // TILE
    a, b = strip_bounds(t, world)[rank]
    r0, r1 = a * TILE, min(b * TILE, n_gene)
    if out is None:
        P = torch.zeros((max(r1 - r0, 1), n_gene), dtype=torch.float64, device=local.slices.device)
        D = torch.zeros_like(P)
    else:
        P, D = out
    if r1 > r0:
        _timed(events, lambda: engine.contract(ctx, MODE_COEX_UPPER, full, full, strip_tiles(t, a, b), dof_a, P, D,
                                               n_products, row0=r0))
    return P, D, full.var[:n_gene], (r0, r1)


def _symm_for(blk, n, n_slices, device, group):
    """Peer-mapped home of this rank's block when TRANSPORT == "ce" (None otherwise).  The barrier
    keeps a rank from overwriting its planes while a peer still pulls the previous call's."""
    if TRANSPORT == "nccl":
        return None
    nbytes = engine.Sliced.storage_bytes(blk, n, n_slices)
    key = (nbytes, torch.device(device).index, id(group))
    if key not in _SYMM:
        try:
            _symm_block(nbytes, device, group)
            ok = 1
        except Exception as e:                      # no peer mapping on this system
            if TRANSPORT == "ce":
                raise
            logging.warning('peer-mapped memory unavailable (%r): NCCL transport', e)
            ok = 0
        flag = torch.tensor([ok], dtype=torch.int32, device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)        # every rank takes the same path
        if int(flag.item()) == 0:
            _SYMM[key] = None
    if _SYMM[key] is None:
        return None
    store, hdl = _SYMM[key]
    hdl.barrier(channel=0, timeout_ms=60000)
    return store, hdl


def coex_sharded(dt_block, dc, n_gene, group=None, precision="default", dimreduce=0, out=None,
                 schedule="pairs", events=None, proj_events=None):
    """Co-expression over all ranks of ``group``.

    dt_block: this rank's genes, rows [rank*blk, min((rank+1)*blk, n_gene)) of the expression
              matrix, blk = row_split(n_gene, world); CUDA float64 (rows_local, n_cell).
    dc:       full covariate matrix (numpy or tensor), identical on all ranks.
    Returns (P_rows, dot_rows, var, (row_begin, row_end)): rows [row_begin, row_end) of P / dot with
    the tiles this rank owns filled in and zeros elsewhere (``owned_tile_mask`` for "pairs"; the
    upper triangle of a strip of tile rows for "allgather"), and var for all genes.
    """
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    ctx = engine.context(dt_block.device)
    n_slices, n_products = engine.PRESETS[precision]
    n = dt_block.shape[1]
    Qt_dev, _, _, dof_a = basis_and_dof(ctx, dc, n, dimreduce)
    blk = row_split(n_gene, world)
    symm = _symm_for(blk, n, n_slices, ctx.device, group) if (schedule == "pairs" and world > 1) else None
    local = _timed(proj_events, lambda: residualize_block(ctx, dt_block, Qt_dev, n_slices, blk,
                                                          storage=None if symm is None else symm[0]))
    if schedule == "allgather":
        return _coex_strip(ctx, local, n_gene, dof_a, n_products, group, out, events)
    P, D, var = _coex_pairs(ctx, local, n_gene, dof_a, n_products, group, out, events, symm=symm)
    return P, D, var, (rank * blk, rank * blk + block_rows(n_gene, world, rank))


def diag_block_streamed(ctx, xh_block, Qt_dev, n_slices, n_products, dof_a, local, out, home, r0):
    """This rank's gene block from the HOST, with its diagonal block of the output done on the way: the rows
    arrive in chunks, each chunk is projected into ``local`` and the tiles of the diagonal block whose columns it
    completes are contracted at once (``association._coex_host_pipeline``), while the next chunk is still on the
    wire and the finished squares leave for ``home`` on a third stream.  The tensor cores would otherwise idle
    until the whole block is in (1 / world of the rank's contraction, and as much of its copy-out, overlap the
    copy-in).  Same bits as the diagonal segment of ``contract_plan``: exact integer sums, symmetric epilogue.
    Returns the event behind the last device->host copy."""
    from .association import _coex_host_pipeline
    rows_a = xh_block.shape[0]
    P, D = out
    local.rows = rows_a
    views = (P[:rows_a, r0:r0 + rows_a], D[:rows_a, r0:r0 + rows_a])
    host = tuple(h[r0:r0 + rows_a, r0:r0 + rows_a] for h in home)
    return _coex_host_pipeline(ctx, xh_block, Qt_dev, n_slices, n_products, dof_a, engine.ENGINE_UMMA, False, host,
                               into=(local, views[0], views[1]))[3]


def coex_host(dt_block_host, dc, n_gene, group=None, precision="default", dimreduce=0, out_dev=None,
              out_host=None, schedule="pairs", home=None):
    """``coex_sharded`` for HOST inputs and outputs: this rank's gene block is a CPU tensor / numpy
    array (pinned memory makes the staged copies asynchronous and overlapped with the projection
    kernels); the rows of P and dot are copied back into ``out_host`` (CPU tensors) if given.
    Returns (P_rows, dot_rows, var, (row_begin, row_end)) as numpy arrays.

    ``home`` = (P, dot) host tensors of the FULL (n_gene, n_gene) matrices ("pairs" schedule): every
    rank writes the rectangles it computed AND their transposes into them.  With tensors from
    ``shared_host_matrices`` (one page-locked mapping shared by all processes) the caller on rank 0
    ends up with what the reference returns to its one caller - the complete symmetric P and dot
    (coex.py:46-48) - once every rank has returned (barrier); P_rows / dot_rows are then None."""
    from .association import _residualize_any
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    ctx = engine.context(None)
    n_slices, n_products = engine.PRESETS[precision]
    xh = dt_block_host if isinstance(dt_block_host, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(dt_block_host))
    n = xh.shape[1]
    Qt_dev, _, _, dof_a = basis_and_dof(ctx, dc, n, dimreduce)
    with torch.cuda.device(ctx.device):
        blk = row_split(n_gene, world)
        symm = _symm_for(blk, n, n_slices, ctx.device, group) if (schedule == "pairs" and world > 1) else None
        local = _own_block(blk, xh.shape[0], n, n_slices, ctx.device, storage=None if symm is None else symm[0])
        tail = None
        streamed = home is not None and schedule == "pairs" and xh.shape[0] > 0 and STREAM_DIAGONAL
        if streamed:
            if out_dev is None:
                out_dev = (torch.zeros((xh.shape[0], n_gene), dtype=torch.float64, device=ctx.device),
                           torch.zeros((xh.shape[0], n_gene), dtype=torch.float64, device=ctx.device))
            tail = diag_block_streamed(ctx, xh, Qt_dev, n_slices, n_products, dof_a, local, out_dev, home, rank * blk)
        elif xh.shape[0]:
            _residualize_any(ctx, xh, Qt_dev, n_slices, False, out=local, row_offset=0)
        if schedule == "allgather":
            P, D, var, (r0, r1) = _coex_strip(ctx, local, n_gene, dof_a, n_products, group, out_dev)
        else:
            P, D, var = _coex_pairs(ctx, local, n_gene, dof_a, n_products, group, out_dev, out_host=out_host, symm=symm,
                                    home=home, skip_diag=streamed)
            r0, r1 = rank * blk, rank * blk + block_rows(n_gene, world, rank)
        if home is not None:
            assert schedule == "pairs"
            torch.cuda.current_stream().synchronize()
            if tail is not None:
                tail.synchronize()
            return None, None, var.cpu().numpy(), (r0, r1)
        if out_host is not None:
            if schedule == "allgather":
                out_host[0].copy_(P, non_blocking=True)
                out_host[1].copy_(D, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            Ph, Dh = out_host[0].numpy(), out_host[1].numpy()
        else:
            Ph, Dh = P.cpu().numpy(), D.cpu().numpy()
        return Ph, Dh, var.cpu().numpy(), (r0, r1)


_SHARED = {}


def shared_host_matrices(count, shape, group=None, tag="nsr"):
    """``count`` float64 host matrices of ``shape`` backed by ONE shared mapping (a file under /dev/shm
    that rank 0 creates and unlinks once everyone has mapped it), page-locked in every process of
    ``group``: all ranks' GPUs copy their parts of a result straight into the same memory, and the
    caller on rank 0 reads the whole of it.  Falls back to private pinned tensors (each process then
    holds only what its own GPU wrote) when /dev/shm is too small; returns (tensors, shared: bool).
    Cached per (count, shape)."""
    import mmap
    import os
    key = (count, tuple(shape), id(group), tag)
    if key in _SHARED:
        return _SHARED[key]
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    each = int(np.prod(shape)) * 8
    nbytes = count * each
    path = [None]
    if rank == 0:
        try:
            free = os.statvfs("/dev/shm")
            if free.f_bavail * free.f_frsize > nbytes + (1 << 28):
                path[0] = "/dev/shm/%s_%d_%d" % (tag, os.getpid(), len(_SHARED))
                with open(path[0], "wb") as f:
                    f.truncate(nbytes)
        except OSError:
            path[0] = None
    if world > 1:
        dist.broadcast_object_list(path, src=0, group=group)
    tensors, shared = None, False
    if path[0] is not None:
        fd = os.open(path[0], os.O_RDWR)
        mm = mmap.mmap(fd, nbytes, mmap.MAP_SHARED, mmap.PROT_READ | mmap.PROT_WRITE)
        os.close(fd)
        flat = torch.frombuffer(mm, dtype=torch.float64)
        if rank == 0:
            flat.zero_()                       # touch the pages once, on the caller's NUMA node
        if world > 1:
            dist.barrier(group=group)
        err = torch.cuda.cudart().cudaHostRegister(flat.data_ptr(), nbytes, 0)
        if int(err) != 0:
            raise RuntimeError("cudaHostRegister of the shared result mapping failed: %r" % (err,))
        if world > 1:
            dist.barrier(group=group)
        if rank == 0:
            os.unlink(path[0])                 # the mapping lives on until every process drops it
        tensors = [flat[i * each // 8:(i + 1) * each // 8].view(*shape) for i in range(count)]
        shared = True
        _SHARED[("mm",) + key] = mm
    else:
        tensors = [torch.empty(tuple(shape), dtype=torch.float64, pin_memory=True) for _ in range(count)]
    _SHARED[key] = (tensors, shared)
    return _SHARED[key]


# ----------------------------------------------------------------------------------------------------
# one process, every GPU of the box: the reference's call, the reference's return value
# ----------------------------------------------------------------------------------------------------
def visible_devices(devices="all"):
    """Normalise a ``devices`` argument ("all", an int count, or a list of device specs) to a list of
    distinct torch.device."""
    if devices is None or devices == "all":
        devices = list(range(torch.cuda.device_count()))
    elif isinstance(devices, int):
        devices = list(range(devices))
    out = []
    for d in devices:
        d = torch.device("cuda", d) if isinstance(d, int) else torch.device(d)
        if d.type != "cuda":
            raise ValueError("devices must be CUDA devices")
        d = torch.device("cuda", torch.cuda.current_device() if d.index is None else d.index)
        if d in out:
            raise ValueError("devices must be distinct (a persistent contraction launch owns its GPU)")
        out.append(d)
    if not out:
        raise RuntimeError("normalisr_b200: no CUDA device visible (there is no CPU fallback).")
    return out


class _Team:
    """What the per-GPU worker threads of one ``coex_all_devices``, ``coexnet_all_devices`` or
    ``coextop_all_devices`` call share."""

    def __init__(self, world):
        import threading
        self.barrier = threading.Barrier(world)
        self.stores = [None] * world          # peer-readable home of every device's block (coextop: its Sliced)
        self.ready = [None] * world           # CUDA event: block residualised
        self.errors = [None] * world
        self.outs = [None] * world            # coexnet: every device's (P, dot) rows, the targets of the peer copies
        self.sent = [None] * world            # CUDA event behind a device's copies to its peers (coextop: its selection)
        self.nets = [None] * world            # coexnet: every device's part of the network (host)
        self.energy = [None] * world          # coextop: every block's digit energies (host)
        self.states = [None] * world          # coextop: every device's partial selection, (G, k, 4) slots


_STORES = {}


def _kept(key, make):
    """``_STORES[key]``, made by ``make()`` on first use: device buffers the worker threads reuse across calls."""
    if key not in _STORES:
        _STORES[key] = make()
    return _STORES[key]


def _device_worker(team, rank, world, dev, xh, dc, n_gene, precision, dimreduce, home, var_out, net=None):
    """One GPU of ``coex_all_devices``, or of ``coexnet_all_devices`` with ``net`` (a ``_NetJob``): then nothing
    goes home; the transposed rectangles go to the peers that own their rows (``contract_plan``'s ``gather``),
    and each device thresholds its complete rows (``_net_rows``)."""
    from .association import _residualize_any
    try:
        torch.cuda.set_device(dev)
        ctx = engine.context(dev)
        n_slices, n_products = engine.PRESETS[precision]
        n = xh.shape[1]
        Qt_dev, _, _, dof_a = basis_and_dof(ctx, dc, n, dimreduce)
        blk = row_split(n_gene, world)
        rows_a = block_rows(n_gene, world, rank)
        r0 = rank * blk
        nbytes = engine.Sliced.storage_bytes(blk, n, n_slices)
        store = _kept((dev.index, "own", nbytes), lambda: torch.empty(nbytes, dtype=torch.uint8, device=dev))
        local = _own_block(blk, rows_a, n, n_slices, dev, storage=store)
        out = _kept((dev.index, "out", max(rows_a, 1), n_gene), lambda: tuple(
            torch.zeros((max(rows_a, 1), n_gene), dtype=torch.float64, device=dev) for _ in range(2)))
        tail = None
        streamed = rows_a > 0 and STREAM_DIAGONAL and net is None       # (streamed: the diagonal block goes home)
        if streamed:
            tail = diag_block_streamed(ctx, xh[r0:r0 + rows_a], Qt_dev, n_slices, n_products, dof_a, local, out, home, r0)
        elif rows_a:
            _residualize_any(ctx, xh[r0:r0 + rows_a], Qt_dev, n_slices, False, out=local, row_offset=0)
        ev = torch.cuda.Event()
        ev.record()
        team.stores[rank], team.ready[rank] = store, ev
        gather = None
        if net is not None:
            team.outs[rank] = out
            gather = team.outs
        team.barrier.wait()                       # every block's event exists
        stores = [_kept((dev.index, d, nbytes), lambda: torch.empty(nbytes, dtype=torch.uint8, device=dev))
                  for d in range(len(exchange_plan(world, rank)))]

        def pull(src, dst):
            torch.cuda.current_stream().wait_event(team.ready[src])
            engine.copy_peer(ctx, dst, team.stores[src])

        rounds = _pull_rounds(ctx, local, rank, world, stores, pull)
        _pairs(ctx, local, rounds, rank, world, n_gene, dof_a, n_products, out, home=home, skip_diag=streamed,
               gather=gather)
        if rows_a:
            var_out[r0:r0 + rows_a].copy_(local.var[:rows_a], non_blocking=True)
        if net is not None:
            _net_rows(ctx, team, rank, world, out, rows_a, r0, net)
        torch.cuda.current_stream().synchronize()
        if tail is not None:
            tail.synchronize()
        team.barrier.wait()                       # nobody still pulls from this device's block
    except BaseException as e:                    # noqa: BLE001 - re-raised by the caller
        team.errors[rank] = e
        team.barrier.abort()


class _NetJob:
    """What ``coexnet_all_devices`` asks of each device: the cutoff, the output form, and where the rows go."""

    def __init__(self, qcut, sparse, edge_values, dense_out):
        self.qcut, self.sparse, self.edge_values, self.dense_out = qcut, sparse, edge_values, dense_out


def _net_rows(ctx, team, rank, world, out, rows_a, r0, job):
    """Once every peer's copies into ``out`` are done, the network of this device's rows [r0, r0 + rows_a):
    team.nets[rank] = (edges, invalid) with the uint8 rows written into job.dense_out, or (indptr, indices[, P_e,
    dot_e]) as numpy arrays of this block's CSR piece."""
    from .binnet import binnet_rows, csr_rows
    main = torch.cuda.current_stream()
    ev = torch.cuda.Event()
    ev.record(main)                               # contract_plan left main behind the copies to the peers
    team.sent[rank] = ev
    team.barrier.wait()                           # every device's event exists
    for s in range(world):
        if s != rank:
            main.wait_event(team.sent[s])
    if not rows_a:
        team.nets[rank] = (0, 0) if not job.sparse else \
            (np.zeros(1, np.int64), np.zeros(0, np.int32)) + ((np.zeros(0), np.zeros(0)) if job.edge_values else ())
        return
    P, D = out[0][:rows_a], out[1][:rows_a]
    stats = torch.zeros(2, dtype=torch.int64, device=P.device)
    if not job.sparse:
        rows, _ = binnet_rows(ctx, P, job.qcut, r0, stats=stats)
        job.dense_out[r0:r0 + rows_a].copy_(rows, non_blocking=True)
        team.nets[rank] = tuple(int(x) for x in stats.cpu())
        return
    piece = csr_rows(ctx, P, job.qcut, r0, stats, D=D if job.edge_values else None)
    team.nets[rank] = tuple(t.cpu().numpy() for t in piece[:4 if job.edge_values else 2])


def _run_team(label, devs, worker, *args):
    """One ``worker(team, rank, world, device, *args)`` thread per GPU; re-raises the first error of any of them
    (a worker that fails records its error in ``team.errors`` and aborts the barrier, releasing the others).
    ``label``: the public entry point, named in the error of a worker stopped at a broken barrier."""
    import threading
    world = len(devs)
    team = _Team(world)
    threads = [threading.Thread(target=worker, name="nsr-gpu%d" % r, args=(team, r, world, devs[r]) + args)
               for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    first = [e for e in team.errors if e is not None and not isinstance(e, threading.BrokenBarrierError)]
    if first:
        raise first[0]
    if any(e is not None for e in team.errors):
        raise RuntimeError("%s: a worker stopped at a broken barrier" % label)
    return team


def _host_f64(dt):
    xh = dt if isinstance(dt, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(dt))
    if xh.is_cuda:
        raise ValueError("coex_all_devices takes a host matrix")
    return xh if xh.dtype == torch.float64 else xh.to(torch.float64)


def coexnet_all_devices(dt, dc, qcut, sparse=False, edge_values=False, devices="all", precision="default",
                        dimreduce=0):
    """``coex.coexnet`` on every GPU of the box from ONE process: the pairs schedule of ``coex_all_devices``,
    but no G x G matrix leaves the GPUs.  Each device ends up holding complete rows of its gene block of P and
    dot (the transposed rectangles of the block pairs travel peer to peer over NVLink), thresholds them with the
    per-row BH kernels and ships its uint8 rows, or its CSR piece, to the host.  Returns (net, var) or, with
    ``edge_values``, (net, var, P_e, dot_e): net a numpy bool (G, G) array or a scipy csr_matrix, exactly
    ``binnet(coex(dt, dc)[0], qcut)`` of one GPU."""
    from .binnet import concat_csr, host_csr
    devs = visible_devices(devices)
    xh = _host_f64(dt)
    n_gene = xh.shape[0]
    dense_out = None if sparse else torch.empty((n_gene, n_gene), dtype=torch.uint8, pin_memory=True)
    var_out = torch.empty(n_gene, dtype=torch.float64, pin_memory=True)
    team = _run_team("coexnet_all_devices", devs, _device_worker, xh, dc, n_gene, precision, dimreduce, None,
                     var_out, _NetJob(qcut, sparse, edge_values, dense_out))
    var = var_out.numpy()
    if not sparse:
        if any(r[1] for r in team.nets):
            raise AssertionError('net must be finite with values in [0, 1].')
        if sum(r[0] for r in team.nets) == 0:
            raise RuntimeError("Empty binary network.")
        return dense_out.numpy().view(bool), var
    parts = concat_csr(team.nets, n_gene)
    if parts[1].size == 0:
        raise RuntimeError("Empty binary network.")
    net = host_csr(n_gene, parts[0], parts[1])
    return (net, var) + tuple(parts[2:])


def coex_all_devices(dt, dc, devices="all", precision="default", dimreduce=0, out=None):
    """``coex`` on every GPU of the box from ONE process: what ``normalisr.coex(dt, dc, devices="all")``
    runs.  One worker thread + stream set per GPU; each residualises its block of genes from the host
    matrix, pulls the digit planes it needs from its peers over NVLink (copy engines), contracts its share
    of the block pairs in one persistent launch and copies every finished rectangle - and its transpose -
    straight into the caller's (n_gene, n_gene) P and dot.  Returns (P, dot, var) as numpy arrays: the
    reference's return value (coex.py:46-48 -> association.py:1036-1057), bit-identical to one GPU.

    dt: (n_gene, n_cell) numpy array or CPU tensor (page-locked memory makes the copies asynchronous);
    out: optional (P, dot) page-locked CPU tensors to fill."""
    devs = visible_devices(devices)
    xh = _host_f64(dt)
    n_gene = xh.shape[0]
    if out is None:
        out = (torch.empty((n_gene, n_gene), dtype=torch.float64, pin_memory=True),
               torch.empty((n_gene, n_gene), dtype=torch.float64, pin_memory=True))
    var_out = torch.empty(n_gene, dtype=torch.float64, pin_memory=True)
    _run_team("coex_all_devices", devs, _device_worker, xh, dc, n_gene, precision, dimreduce, out, var_out)
    return out[0].numpy(), out[1].numpy(), var_out.numpy()


TopDeal = collections.namedtuple("TopDeal", "a b lo hi pulls parts")
TopDeal.__doc__ = """One GPU's share of ``coextop_all_devices``: the strips of tile rows [a, b) it selects over; the
rows [lo, hi) of its gene block, which it residualises and whose final lists it merges; ``pulls``, the blocks it
copies from their owners (every other block with rows in [a * TILE, G), the rows its strips read; none for an
empty range); ``parts``, the ranks whose selections reach rows of its block (a non-empty range starting below
hi: their merge parts)."""


def coextop_deal(n_gene, world):
    """[TopDeal] per rank: tile rows dealt out with ``strip_bounds`` (equal numbers of upper tiles, so the
    contraction and the selection are balanced alike), gene blocks with ``row_split``.  A pair (i < j) lies in
    the strip of row i and reaches rows i and j there; the GPU owning that strip touches only rows >= its first
    strip row, which is what ``pulls`` and ``parts`` follow from."""
    t = (n_gene + TILE - 1) // TILE
    blk = row_split(n_gene, world)
    spans = [(d * blk, d * blk + block_rows(n_gene, world, d)) for d in range(world)]
    ranges = strip_bounds(t, world)
    deal = []
    for r in range(world):
        (a, b), (lo, hi) = ranges[r], spans[r]
        pulls = [d for d in range(world) if d != r and b > a and spans[d][1] > max(spans[d][0], a * TILE)]
        parts = [w for w in range(world) if hi > lo and ranges[w][1] > ranges[w][0] and ranges[w][0] * TILE < hi]
        deal.append(TopDeal(a, b, lo, hi, pulls, parts))
    return deal


def _top_worker(team, rank, world, dev, xh, dc, n_gene, k, precision, dimreduce, out):
    """One GPU of ``coextop_all_devices``: residualise its block into a full G-row Sliced, pull the blocks its
    strips read from their owners, select over its strips on a reset state, then merge the partial lists of its
    block's rows from every GPU that touched them and copy the result into ``out`` = (idx, P_k, dot_k, var)."""
    from .association import _residualize_any
    from .coex import top_strips
    try:
        torch.cuda.set_device(dev)
        ctx = engine.context(dev)
        n_slices, n_products = engine.PRESETS[precision]
        n = xh.shape[1]
        Qt_dev, _, _, dof_a = basis_and_dof(ctx, dc, n, dimreduce)
        deal = coextop_deal(n_gene, world)
        me = deal[rank]
        main = torch.cuda.current_stream()
        full = engine.Sliced(n_gene, n, n_slices, dev)
        if me.hi > me.lo:
            _residualize_any(ctx, xh[me.lo:me.hi], Qt_dev, n_slices, False, out=full, row_offset=me.lo)
        ev = torch.cuda.Event()
        ev.record()
        team.stores[rank], team.ready[rank] = full, ev
        team.energy[rank] = full.energy_max.cpu().numpy()
        team.barrier.wait()                       # every block's event and energies exist
        for d in me.pulls:
            lo, hi, src = deal[d].lo, deal[d].hi, team.stores[d]
            main.wait_event(team.ready[d])
            for s in range(n_slices):
                engine.copy_peer(ctx, full.slices[s, lo:hi], src.slices[s, lo:hi])
            engine.copy_peer(ctx, full.quantum[lo:hi], src.quantum[lo:hi])
            engine.copy_peer(ctx, full.var[lo:hi], src.var[lo:hi])
        em = np.maximum.reduce(team.energy)       # NaN (non-finite input) propagates
        k_chunk = engine.plan_k_chunk(full, full, n_products, energies=(em, em))
        state = torch.empty((n_gene, k, 4), dtype=torch.float64, device=dev)
        engine.topk_reset(ctx, state)
        top_strips(ctx, full, dof_a, n_products, k_chunk, state, me.a, me.b)
        ev = torch.cuda.Event()
        ev.record()
        team.sent[rank], team.states[rank] = ev, state
        team.barrier.wait()                       # every selection's event exists
        if me.hi > me.lo:
            parts = []
            for w in me.parts:
                if w == rank:
                    parts.append(state[me.lo:me.hi])
                    continue
                main.wait_event(team.sent[w])
                parts.append(torch.empty((me.hi - me.lo, k, 4), dtype=torch.float64, device=dev))
                engine.copy_peer(ctx, parts[-1], team.states[w][me.lo:me.hi])
            res = engine.topk_merge(ctx, parts) + (full.var[me.lo:me.hi],)
            for t, o in zip(res, out):
                o[me.lo:me.hi].copy_(t, non_blocking=True)
        main.synchronize()
        team.barrier.wait()                       # nobody still copies from this device's planes or state
    except BaseException as e:                    # noqa: BLE001 - re-raised by the caller
        team.errors[rank] = e
        team.barrier.abort()


def coextop_all_devices(dt, dc, k, devices="all", precision="default", dimreduce=0):
    """``coex.coextop`` on every GPU of the box from ONE process: the strips of tile rows are dealt out
    (``coextop_deal``), every GPU keeps a partial top k for each row over its strips, and the owner of each
    gene block merges the partial lists of its rows (``nsr_topk_merge``).  The ranking order is total and the
    sums are exact, so the result is bit-identical to one GPU.  dt: (n_gene, n_cell) numpy array or CPU tensor
    (k already checked by ``coextop``).  Returns (idx, P_k, dot_k, var) as numpy arrays."""
    devs = visible_devices(devices)
    if len(devs) > TOPK_MAX_PARTS:
        raise ValueError("coextop takes at most %d devices" % TOPK_MAX_PARTS)
    xh = _host_f64(dt)
    n_gene = xh.shape[0]
    out = (torch.empty((n_gene, k), dtype=torch.int64, pin_memory=True),
           torch.empty((n_gene, k), dtype=torch.float64, pin_memory=True),
           torch.empty((n_gene, k), dtype=torch.float64, pin_memory=True),
           torch.empty(n_gene, dtype=torch.float64, pin_memory=True))
    _run_team("coextop_all_devices", devs, _top_worker, xh, dc, n_gene, k, precision, dimreduce, out)
    return tuple(t.numpy() for t in out)


def de_all_devices(dx, dy, dc, devices="all", **ka):
    """``association_tests(dx, dy, dc, ...)`` (dy given: DE, any ``single``) with the rows of dy - the genes -
    dealt out to the GPUs of this process, one worker thread per GPU, no exchange at all (SURVEY 8e: dg and
    dc are small and replicated; every test is independent in y).  Host inputs, host outputs with the
    reference's shapes: the per-device results are concatenated along the gene axis."""
    import threading
    from .association import association_tests
    devs = visible_devices(devices)
    world = len(devs)
    ny = dy.shape[0]
    blk = row_split(ny, world)
    spans = [(k * blk, min((k + 1) * blk, ny)) for k in range(world) if k * blk < ny]
    res, err = [None] * len(spans), [None] * len(spans)

    def work(k):
        try:
            torch.cuda.set_device(devs[k])
            res[k] = association_tests(dx, dy[spans[k][0]:spans[k][1]], dc, device=devs[k], **ka)
        except BaseException as e:                # noqa: BLE001 - re-raised by the caller
            err[k] = e

    threads = [threading.Thread(target=work, args=(k,), name="nsr-gpu%d" % k) for k in range(len(spans))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for e in err:
        if e is not None:
            raise e
    P = np.concatenate([r[0] for r in res], axis=1)
    out2 = np.concatenate([r[1] for r in res], axis=1)
    alpha = None if res[0][2] is None else np.concatenate([r[2] for r in res], axis=1)
    vary = np.concatenate([r[4] for r in res], axis=-1)
    return P, out2, alpha, res[0][3], vary


def block_spans(n_gene, world, schedule="pairs"):
    """Global row range [r0, r1) every rank's output rows cover (same ``schedule`` as coex_sharded)."""
    t = (n_gene + TILE - 1) // TILE
    if schedule == "allgather":
        return [(a * TILE, min(b * TILE, n_gene)) for a, b in strip_bounds(t, world)]
    blk = row_split(n_gene, world)
    return [(k * blk, k * blk + block_rows(n_gene, world, k)) for k in range(world)]


def assemble_dense(row_blocks, n_gene, world, schedule="pairs"):
    """Full symmetric (n_gene, n_gene) matrix from the per-rank outputs of ``coex_sharded`` /
    ``_coex_pairs``: ``row_blocks[k]`` holds rank k's rows (tiles it owns filled in, zeros elsewhere).
    Entry (i, j) was computed by the owner of tile (i, j) or, mirrored, of tile (j, i); this is the
    one assembly rule, shared by ``gather_dense`` (multi-process), ``coex_all_devices`` (one process)
    and the one-GPU emulation of the schedule in the tests."""
    spans = block_spans(n_gene, world, schedule)
    dev = row_blocks[0].device
    full = torch.zeros((n_gene, n_gene), dtype=torch.float64, device=dev)
    for (r0, r1), blk_t in zip(spans, row_blocks):
        if r1 > r0:
            full[r0:r1] = blk_t[:r1 - r0].to(dev)
    if schedule == "allgather":
        up = torch.triu(full, 1)
        return up + up.T
    res = torch.empty_like(full)
    for k, (r0, r1) in enumerate(spans):
        if r1 <= r0:
            continue
        m = torch.from_numpy(owned_tile_mask(n_gene, world, k)).to(dev)
        m = m.repeat_interleave(TILE, 0)[:r1 - r0].repeat_interleave(TILE, 1)[:, :n_gene]
        res[r0:r1] = torch.where(m, full[r0:r1], full[:, r0:r1].T)
    return res


def gather_dense(P_rows, D_rows, bounds, n_gene, group=None, dst=0, schedule="pairs"):
    """Assemble the full symmetric (n_gene, n_gene) P and dot on rank ``dst`` (None elsewhere)
    from the per-rank outputs of ``coex_sharded`` (same ``schedule``)."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    dev = P_rows.device
    spans = block_spans(n_gene, world, schedule)
    outs = []
    for src_t in (P_rows, D_rows):
        blocks = []
        for k, (r0, r1) in enumerate(spans):
            if r1 <= r0:
                blocks.append(torch.empty((0, n_gene), dtype=torch.float64, device=dev))
            elif k == dst:
                blocks.append(src_t[:r1 - r0] if rank == dst else None)
            elif rank == dst:
                buf = torch.empty((r1 - r0, n_gene), dtype=torch.float64, device=dev)
                dist.recv(buf, src=k, group=group)
                blocks.append(buf)
            else:
                if rank == k:
                    dist.send(src_t[:r1 - r0].contiguous(), dst=dst, group=group)
                blocks.append(None)
        outs.append(assemble_dense(blocks, n_gene, world, schedule) if rank == dst else None)
    return outs[0], outs[1]


def de_sharded(dg, dt_block, dc, n_gene, group=None, precision="default", dimreduce=0):
    """DE (single=0) with genes sharded over ranks: no exchange step at all (dg and dc are small
    and replicated).  Returns (P, gamma, varg, vart_block) for this rank's genes."""
    ctx = engine.context(dt_block.device)
    n_slices, n_products = engine.PRESETS[precision]
    n = dt_block.shape[1]
    Qt_dev, crank, _ = covariate_basis_device(ctx, dc)
    A = engine.residualize(ctx, dg.to(ctx.device, torch.float64), Qt_dev, n_slices)
    B = engine.residualize(ctx, dt_block, Qt_dev, n_slices)
    P = torch.empty((A.rows, B.rows), dtype=torch.float64, device=ctx.device)
    G = torch.empty_like(P)
    engine.contract(ctx, MODE_DE, A, B, engine.rect_tiles(A.rows, B.rows), (n - 1 - crank - dimreduce) / 2,
                    P, G, n_products)
    return P, G, A.var, B.var
