"""Page-locked staging between a caller's ordinary (pageable) host arrays and the device.

The copy engines only run asynchronously - and at full PCIe rate - on page-locked memory.  The reference's callers
hold plain numpy arrays (``coex.py:4``: ``dt``, ``dc`` in, fresh ``P``, ``dot`` out), and a pageable ``cudaMemcpy``
stages through one driver thread at ~3 GB/s and takes the page faults of a fresh result array one by one:
``norm.coex(dt, dc)`` on numpy arrays took 4.4 - 5.4 s at 100k cells x 20k genes where page-locked buffers take
0.32 s.  Here a team of host threads (``nsr_host_copy2d``) moves the data between the caller's arrays and small
rings of page-locked slots, so that the plain call runs the same three-stream pipeline:

    InputStager   rows of a host matrix -> device buffer (direct when the matrix is page-locked already)
    OutputDrain   blocks of device matrices -> pageable host matrices, drained by a worker thread
"""
import queue
import threading

import torch

from . import _lib

STAGE_BYTES = 1 << 28      # row blocks of the host loops: each is staged through page-locked slots of this size
_SLOTS = {}        # (tag, device index, bytes, count) -> list of page-locked uint8 tensors, kept for the next call


def host_copy2d(dst, src, threads=0):
    """dst <- src for 2-D CPU tensors of equal shape and dtype with unit column stride, by a team of threads."""
    assert dst.shape == src.shape and dst.dtype == src.dtype and dst.dim() == 2
    assert (dst.shape[1] <= 1 or (dst.stride(1) == 1 and src.stride(1) == 1))
    rows, cols = dst.shape
    if rows == 0 or cols == 0:
        return
    es = dst.element_size()
    dp = dst.stride(0) * es if rows > 1 else cols * es
    sp = src.stride(0) * es if rows > 1 else cols * es
    _lib.check(_lib.load().nsr_host_copy2d(dst.data_ptr(), dp, src.data_ptr(), sp, cols * es, rows, int(threads)),
               "nsr_host_copy2d")


def pinned_slots(tag, device, nbytes, count):
    """``count`` page-locked buffers of at least ``nbytes`` for one purpose and device; a ring that is large enough
    is reused by later calls (page-locking memory costs about as much time as copying it once)."""
    nbytes = -(-int(nbytes) // (1 << 20)) * (1 << 20)
    head = (tag, torch.device(device).index, count)
    for k in list(_SLOTS):
        if k[:3] == head:
            if k[3] >= nbytes:
                return _SLOTS[k]
            del _SLOTS[k]                                        # outgrown
    _SLOTS[head + (nbytes,)] = [torch.empty(nbytes, dtype=torch.uint8, pin_memory=True) for _ in range(count)]
    return _SLOTS[head + (nbytes,)]


def release():
    """Give the page-locked rings back (they are otherwise kept for the next call: up to ~1.5 GB per device)."""
    _SLOTS.clear()


def to_device(ctx, src, tag="flat"):
    """A 1-D host tensor -> a new device tensor on the current stream, through the page-locked slots: the array is
    taken as rows of 1 MB (and a shorter last row), at most STAGE_BYTES per slot.  Returns once the slots are free
    again (the copies out of them are done), so the next call may use the same tag."""
    n, es = src.numel(), src.element_size()
    dst = torch.empty(max(1, n), dtype=src.dtype, device=ctx.device)[:n]
    stream = torch.cuda.current_stream(ctx.device)
    width = max(1, min(n, (1 << 20) // es))
    rows = n // width
    if rows:
        step = max(1, min(rows, STAGE_BYTES // (width * es)))
        stager = InputStager(src[:rows * width].view(rows, width), step, ctx.device, tag=tag)
        for r0 in range(0, rows, step):
            r1 = min(rows, r0 + step)
            stager.copy_rows(dst[r0 * width:r1 * width].view(r1 - r0, width), r0, r1, stream)
        stager.wait()
    if rows * width < n:
        tail = src[rows * width:].view(1, n - rows * width)
        stager = InputStager(tail, 1, ctx.device, tag=tag + "-tail")
        stager.copy_rows(dst[rows * width:].view(tail.shape), 0, 1, stream)
        stager.wait()
    return dst


class InputStager:
    """Rows [r0, r1) of a 2-D host matrix (any dtype) -> a device buffer of the same dtype, asynchronously on a
    stream."""

    def __init__(self, src, rows_max, device, tag="in"):
        self.src = src
        self.pinned = src.is_pinned()
        self.k = 0
        if not self.pinned:
            n, es = src.shape[1], src.element_size()
            self.slots = [s[:rows_max * n * es].view(src.dtype).view(rows_max, n)
                          for s in pinned_slots(tag, device, max(1, rows_max * n * es), 2)]
            self.events = [None, None]

    def copy_rows(self, dst_dev, r0, r1, stream):
        """dst_dev[:r1 - r0] <- src[r0:r1] on ``stream``.  Page-locked source: one asynchronous copy.  Pageable
        source: the rows go into a page-locked slot first (thread team; waits for the copy that last used the
        slot), the slot is copied asynchronously."""
        if self.pinned:
            with torch.cuda.stream(stream):
                dst_dev[:r1 - r0].copy_(self.src[r0:r1], non_blocking=True)
            return
        i = self.k & 1
        self.k += 1
        if self.events[i] is not None:
            self.events[i].synchronize()
        slot = self.slots[i][:r1 - r0]
        rows = self.src[r0:r1]
        if rows.shape[1] <= 1 or rows.stride(1) == 1:
            host_copy2d(slot, rows)
        else:
            slot.copy_(rows)                       # other dtypes / column strides: torch's own (converting) copy
        with torch.cuda.stream(stream):
            dst_dev[:r1 - r0].copy_(slot, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(stream)
        self.events[i] = ev

    def wait(self):
        """Until the copies out of the page-locked slots are done."""
        for ev in (self.events if not self.pinned else ()):
            if ev is not None:
                ev.synchronize()


class OutputDrain:
    """Blocks of device matrices -> pageable host matrices: each ``send`` queues device->host copies of its blocks
    into one page-locked slot on the given stream; a worker thread waits for them and copies the slot out with the
    thread team (the first-touch page faults of a fresh result array are spread over all cores), then frees it."""

    def __init__(self, ctx, slot_bytes, count=3, tag="out"):
        self.ctx = ctx
        self.slots = pinned_slots(tag, ctx.device, slot_bytes, count)
        self.slot_bytes = self.slots[0].numel()
        self.free = queue.Queue()
        for i in range(count):
            self.free.put(i)
        self.jobs = queue.Queue()
        self.error = None
        self.thread = threading.Thread(target=self._run, name="nsr-drain", daemon=True)
        self.thread.start()

    def send(self, stream, blocks):
        """blocks: list of (dst host 2-D view, src device 2-D view) of equal shapes and dtypes (unit column stride)."""
        batch, used = [], 0
        for dst, src in blocks:
            rows, cols = src.shape
            if rows == 0 or cols == 0:
                continue
            es = src.element_size()
            rows_fit = max(1, self.slot_bytes // (cols * es))
            for a in range(0, rows, rows_fit):                 # a block larger than a slot goes in row pieces
                b = min(rows, a + rows_fit)
                nb = -(-((b - a) * cols * es) // 16) * 16       # keep every piece 16-byte aligned in the slot
                if used + nb > self.slot_bytes and batch:
                    self._flush(stream, batch)
                    batch, used = [], 0
                batch.append((dst[a:b], src[a:b], nb))
                used += nb
        if batch:
            self._flush(stream, batch)

    def _flush(self, stream, batch):
        i = self.free.get()                                    # blocks while every slot is in flight
        if self.error is not None:
            self.free.put(i)
            raise self.error
        slot, off, parts = self.slots[i], 0, []
        lib = self.ctx.lib
        for dst, src, nb in batch:
            rows, cols = src.shape
            es = src.element_size()
            stage = slot[off:off + rows * cols * es].view(src.dtype).view(rows, cols)
            _lib.check(lib.nsr_copy2d(self.ctx.handle, stream.cuda_stream, stage.data_ptr(), cols * es, src.data_ptr(),
                                      (src.stride(0) if rows > 1 else cols) * es, cols * es, rows, 0), "nsr_copy2d")
            parts.append((dst, stage))
            off += nb
        ev = torch.cuda.Event()
        ev.record(stream)
        self.jobs.put((i, ev, parts))

    def _run(self):
        while True:
            job = self.jobs.get()
            if job is None:
                return
            i, ev, parts = job
            try:
                ev.synchronize()
                for dst, stage in parts:
                    host_copy2d(dst, stage)
            except BaseException as e:          # noqa: BLE001 - re-raised by close()
                self.error = e
            self.free.put(i)

    def close(self):
        """Wait until everything sent has reached the host matrices."""
        self.jobs.put(None)
        self.thread.join()
        if self.error is not None:
            raise self.error


class RowBlocks:
    """The row-block loop of the functions around the hot path (normvar, lcpm, compute_var, binnet) on HOST
    matrices: ``fetch(g0, g1)`` returns rows [g0, g1) of the source on the device (pageable sources through the
    page-locked slots), ``store(dst_rows, res_dev)`` sends a result block to its rows of a pageable host matrix
    through the drain, ``close()`` waits for everything."""

    def __init__(self, ctx, src, rows_max, out_row_bytes=0, tag="blocks"):
        self.ctx = ctx
        self.src = src                     # None: results only (the source is on the device already)
        self.stager = InputStager(src, rows_max, ctx.device, tag=tag + "-in") if src is not None else None
        self.drain = OutputDrain(ctx, max(1 << 20, rows_max * out_row_bytes), count=2, tag=tag + "-out") \
            if out_row_bytes else None

    def fetch(self, g0, g1):
        dst = torch.empty((g1 - g0, self.src.shape[1]), dtype=self.src.dtype, device=self.ctx.device)
        self.stager.copy_rows(dst, g0, g1, torch.cuda.current_stream(self.ctx.device))
        return dst

    def store(self, dst_rows, res_dev):
        self.drain.send(torch.cuda.current_stream(self.ctx.device), [(dst_rows, res_dev)])

    def close(self):
        if self.drain is not None:
            self.drain.close()
