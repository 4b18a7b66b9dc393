"""Host-side logic of the multi-GPU path on CPU: strip partition, tile lists, and the
all-gather of digit planes over a world_size-2 gloo group."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from normalisr_b200 import engine, parallel


@pytest.mark.parametrize("world", [1, 2, 4, 8])
@pytest.mark.parametrize("rows", [100, 1000, 5000, 20000])
def test_strips_partition_upper_triangle(rows, world):
    t = (rows + 127) // 128
    strips = parallel.strip_bounds(t, world)
    assert len(strips) == world and strips[0][0] == 0 and strips[-1][1] == t
    seen = set()
    counts = []
    for a, b in strips:
        tl = parallel.strip_tiles(t, a, b)
        counts.append(len(tl))
        for x in map(tuple, tl):
            assert x not in seen and a <= x[0] < b and x[0] <= x[1]
            seen.add(x)
    assert len(seen) == t * (t + 1) // 2
    if t >= 8 * world:
        assert max(counts) <= 1.25 * (sum(counts) / world) + t      # balanced up to one tile row


@pytest.mark.parametrize("rows", [130, 1900, 5000, 20000])
@pytest.mark.parametrize("world", [1, 2, 3, 4, 5, 8])
def test_home_rectangles_write_every_entry_exactly_once(rows, world):
    """The single-caller result: every rank copies home its diagonal block (both triangles, the lower one from
    the kernel's mirrored stores), and for every block pair it owns the rectangle it computed plus the
    transpose.  Together these must cover the (rows x rows) matrices exactly once - no entry left to a
    second pass on the host, none written by two GPUs - and each rectangle must consist of whole tiles the
    rank really computes (``pair_tiles``)."""
    blk = parallel.row_split(rows, world)
    count = np.zeros((rows, rows), dtype=np.int32)
    for rank in range(world):
        ra = parallel.block_rows(rows, world, rank)
        r0 = rank * blk
        if not ra:
            continue
        count[r0:r0 + ra, r0:r0 + ra] += 1
        for _, src, parity in parallel.exchange_plan(world, rank):
            rb = parallel.block_rows(rows, world, src)
            if not rb:
                continue
            c0 = src * blk
            a0, a1, b0, b1 = parallel._segment_rect(ra, rb, parity)
            count[r0 + a0:r0 + a1, c0 + b0:c0 + b1] += 1                 # direct
            count[c0 + b0:c0 + b1, r0 + a0:r0 + a1] += 1                 # transposed copy
            tl = parallel.pair_tiles(ra, rb, parity)
            cover = np.zeros((ra, rb), dtype=bool)
            for ti, tj in tl:
                cover[ti * 128:(ti + 1) * 128, tj * 128:(tj + 1) * 128] = True
            want = np.zeros((ra, rb), dtype=bool)
            want[a0:a1, b0:b1] = True
            assert np.array_equal(cover, want)
    assert (count == 1).all()


@pytest.mark.parametrize("rows", [130, 1900, 5000, 20000])
@pytest.mark.parametrize("world", range(1, 9))
@pytest.mark.parametrize("mirrored", [False, True])
def test_segment_plan_covers_every_entry_exactly_once(rows, world, mirrored):
    """The segments ``contract_plan`` launches, as ``plan_segments`` builds them (block pairs cut into column
    strips when the transposes are written): their rects and the transposes of them cover the (rows x rows)
    matrix exactly once, the diagonal block's upper-triangular tiles and their transposes cover its square,
    and every block pair's tiles cover exactly its rect."""
    blk = parallel.row_split(rows, world)
    count = np.zeros((rows, rows), dtype=np.int32)
    for rank in range(world):
        rounds = [(src, parity, None, []) for _, src, parity in parallel.exchange_plan(world, rank)]
        segs = parallel.plan_segments(rounds, rank, world, rows, mirrored=mirrored)
        ra, r0 = parallel.block_rows(rows, world, rank), rank * blk
        assert len(segs) <= parallel.MAX_SEGMENTS and (ra > 0 or not segs)
        for sg in segs:
            a0, a1, b0, b1 = sg.rect
            rb, c0 = parallel.block_rows(rows, world, sg.src), sg.col0
            assert c0 == sg.src * blk and sg.rows_b == rb and sg.tiles.dtype == np.int32
            cover = np.zeros((ra, rb), dtype=bool)
            for ti, tj in sg.tiles:
                cover[ti * 128:(ti + 1) * 128, tj * 128:(tj + 1) * 128] = True
            if sg.diagonal:
                assert sg.src == rank and sg.k == 0 and sg.rect == (0, ra, 0, ra)
                cover |= cover.T
                count[r0:r0 + ra, r0:r0 + ra] += 1
            else:
                assert rounds[sg.k - 1][0] == sg.src
                count[r0 + a0:r0 + a1, c0 + b0:c0 + b1] += 1                # direct
                count[c0 + b0:c0 + b1, r0 + a0:r0 + a1] += 1                # transposed copy
            want = np.zeros((ra, rb), dtype=bool)
            want[a0:a1, b0:b1] = True
            assert np.array_equal(cover, want)
        if mirrored and world > 2 and rows >= 5000:
            assert len(segs) > 1 + len(rounds)                          # block pairs leave in strips
    assert (count == 1).all()


@pytest.mark.parametrize("rows_a,rows_b,parity", [(2560, 2560, None), (2560, 2440, 0), (2500, 2560, 1), (130, 100, None),
                                                  (10000, 10000, 0), (128, 128, 1)])
@pytest.mark.parametrize("n_sub", [1, 2, 4, 8, 50])
def test_pair_strips_partition_tiles_and_columns(rows_a, rows_b, parity, n_sub):
    """Column strips of a block pair (each leaves for the host as soon as it is contracted): together they hold
    every tile of the pair once, in the original order within a strip, and their rectangles tile the pair's
    rectangle without gaps or overlaps, each rectangle covered by its own tiles."""
    tl = parallel.pair_tiles(rows_a, rows_b, parity)
    rect = parallel._segment_rect(rows_a, rows_b, parity)
    strips = parallel.pair_strips(tl, rect, n_sub)
    assert 1 <= len(strips) <= max(1, n_sub)
    assert sorted(map(tuple, np.concatenate([t for t, _ in strips]))) == sorted(map(tuple, tl))
    a0, a1, b0, b1 = rect
    if not len(tl):                                   # the other owner took the only tile row / column
        assert strips[0][1] == rect and (a1 - a0) * (b1 - b0) == 0
        return
    count = np.zeros((rows_a, rows_b), dtype=np.int32)
    for tiles, (s0, s1, c0, c1) in strips:
        assert (s0, s1) == (a0, a1) and b0 <= c0 < c1 <= b1
        count[s0:s1, c0:c1] += 1
        cover = np.zeros((rows_a, rows_b), dtype=bool)
        for ti, tj in tiles:
            cover[ti * 128:(ti + 1) * 128, tj * 128:(tj + 1) * 128] = True
        assert cover[s0:s1, c0:c1].all()
        order = [tuple(x) for x in tl if c0 <= x[1] * 128 < c1]
        assert [tuple(x) for x in tiles] == order
    assert (count[a0:a1, b0:b1] == 1).all() and count.sum() == (a1 - a0) * (b1 - b0)


def test_row_split():
    # equal blocks, multiples of the 128-row tile
    assert parallel.row_split(20000, 8) == 2560 and parallel.row_split(10, 4) == 128
    assert parallel.row_split(20000, 1) == 20096
    assert [parallel.block_rows(20000, 8, k) for k in (0, 6, 7)] == [2560, 2560, 2080]
    assert [parallel.block_rows(300, 4, k) for k in range(4)] == [128, 128, 44, 0]


@pytest.mark.parametrize("world", [1, 2, 3, 4, 5, 8])
@pytest.mark.parametrize("rows", [100, 300, 1000, 5000, 20000])
def test_pairs_schedule_covers_every_tile_pair_once(rows, world):
    """Circulant block-pair schedule: every unordered tile pair is computed by exactly one rank,
    each rank receives world // 2 blocks, work is balanced, rounds are mutually consistent."""
    t = (rows + 127) // 128
    tb = parallel.row_split(rows, world) // 128
    cnt = np.zeros((t, t), dtype=int)
    work = []
    for r in range(world):
        plan = parallel.exchange_plan(world, r)
        assert len(plan) == world // 2
        for d, (dst, src, parity) in enumerate(plan, 1):
            assert src == (r + d) % world and dst == (r - d) % world
            # my round-d receive is my source's round-d send
            assert parallel.exchange_plan(world, src)[d - 1][0] == r
            if parity is not None:
                other = [p for (_, s2, p) in parallel.exchange_plan(world, src) if s2 == r]
                assert other == [1 - parity]
        m = parallel.owned_tile_mask(rows, world, r)
        work.append(int(m.sum()))
        for i, j in zip(*np.nonzero(m)):
            gi = r * tb + i
            cnt[min(gi, j), max(gi, j)] += 1
    assert (cnt[np.triu_indices(t)] == 1).all()
    if t >= 16 * world:
        assert max(work) <= 1.06 * sum(work) / world


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, rows_total, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        blk = parallel.row_split(rows_total, world)
        local = engine.Sliced(blk, 200, 3, "cpu")
        g = torch.Generator().manual_seed(100 + rank)
        local.slices.copy_(torch.randint(-128, 128, local.slices.shape, generator=g, dtype=torch.int8))
        local.quantum.fill_(rank + 1.0)
        local.var.fill_(10.0 * (rank + 1))
        # block exchange of the pairs schedule: round d brings block (rank + d) % world
        for src, parity, buf, works in parallel.start_exchange(local):
            parallel.wait_block(works)
            gk = torch.Generator().manual_seed(100 + src)
            want = torch.randint(-128, 128, local.slices.shape, generator=gk, dtype=torch.int8)
            if not (torch.equal(buf.slices, want) and bool((buf.quantum == src + 1.0).all())
                    and bool((buf.var == 10.0 * (src + 1)).all())):
                q.put((rank, False))
                return
        full = parallel.gather_sliced(local, rows_total)
        ok = full.rows == rows_total and full.rows_alloc == blk * world
        for k in range(world):
            gk = torch.Generator().manual_seed(100 + k)
            want = torch.randint(-128, 128, local.slices.shape, generator=gk, dtype=torch.int8)
            ok = ok and torch.equal(full.slices[:, k * blk:(k + 1) * blk], want)
            ok = ok and bool((full.quantum[k * blk:(k + 1) * blk] == k + 1.0).all())
            ok = ok and bool((full.var[k * blk:(k + 1) * blk] == 10.0 * (k + 1)).all())
        # assembly of the full symmetric matrices from the rows each rank owns (pairs schedule)
        for total in (rows_total, 300, 700):
            gen = torch.Generator().manual_seed(7)
            F = torch.rand((total, total), generator=gen, dtype=torch.float64)
            F = torch.triu(F, 1)
            F = F + F.T
            b = parallel.row_split(total, world)
            r0, r1 = rank * b, rank * b + parallel.block_rows(total, world, rank)
            m = torch.from_numpy(parallel.owned_tile_mask(total, world, rank))
            m = m.repeat_interleave(128, 0)[:max(r1 - r0, 0)].repeat_interleave(128, 1)[:, :total]
            mine = torch.where(m, F[r0:r1], torch.zeros_like(F[r0:r1])) if r1 > r0 else torch.zeros((1, total), dtype=torch.float64)
            Pf, Df = parallel.gather_dense(mine, 2 * mine, None, total)
            if rank == 0:
                ok = ok and torch.equal(Pf, F) and torch.equal(Df, 2 * F)
        q.put((rank, bool(ok)))
    finally:
        dist.destroy_process_group()


def test_gather_sliced_gloo_world2():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, 37, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True)]
