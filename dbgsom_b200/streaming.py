"""Fits whose samples do not fit in device memory: chunk planning and the pinned host staging ring.

When the resident fit (every sample, its fp16 shadows and the per-sample buffers of the search, K2 and the
post-training passes in HBM) would not fit in free device memory, `DeviceEngine` keeps only per-sample vectors on
the device and streams the rows from the user's host array in chunks, every epoch.  `plan_stream` decides which of
the two a fit takes and how large the chunks are; `HostStager` moves the rows through a fixed ring of page-locked
buffers.  DESIGN.md, "Streaming fits", describes the pipeline.
"""

from __future__ import annotations

import collections
import contextlib
import os
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from typing import Callable

import numpy as np

ROW_GRANULE = 256                 # chunk row counts are multiples of this
MAX_CHUNK_BYTES = 512 << 20       # float32 rows of one planned chunk (the first chunk's copy is not hidden)
RING_PIECES = 8                   # page-locked staging buffers ...
RING_PIECE_BYTES = 128 << 20      # ... of at most this size each: the ring holds at most 1 GiB


def _round_up(a: int, b: int) -> int:
    return (a + b - 1) // b * b


def free_margin(total_bytes: int) -> int:
    """Device bytes the planner leaves unused: 2 GiB or 1/32 of the card, whichever is larger (allocator
    fragmentation, the smoothing workspace, cuBLAS/NCCL buffers and the CUDA context's own growth)."""
    return max(2 << 30, int(total_bytes) // 32)


def _map_bytes(capacity: int, ldx: int, ld16: int, n_classes: int, streamed: bool) -> int:
    """Map buffers at capacity: two float64 prototype copies, the float32 copy, the fp16 shadows, the epoch sums
    `part`, the M^2 uint16 hop matrix and the class histogram; a streamed fit holds one more `part` and histogram
    for the chunk it is summing."""
    cap = _round_up(max(int(capacity), 4), 256)
    part = (cap * ldx + 3 * cap) * 8
    hist = cap * n_classes * 8
    b = 2 * cap * ldx * 8 + cap * ldx * 4 + 2 * cap * ld16 * 2 + cap * (64 * 2 + 4 + 8) + part + cap * cap * 2 + hist
    return b + (part + hist if streamed else 0)


def _widths(d: int) -> tuple[int, int]:
    ldx = _round_up(int(d), 4)
    return ldx, _round_up(ldx, 64)


def resident_bytes(n: int, d: int, capacity: int, n_classes: int, weighted: bool,
                   acc_ws_bytes: Callable[[int, int, int], int], bmu_ws_bytes: Callable[[int, int], int]) -> int:
    """Device bytes the resident fit allocates: X float32 [N, ldx], the hi/lo fp16 shadows and xnorm16, the
    shadow-row permutation, the epoch winners [N, 2], the post-training winners and distances [N, 2], labels and
    weights, the K2 and BMU workspaces for N rows, and the map buffers at capacity."""
    ldx, ld16 = _widths(d)
    cap = _round_up(max(int(capacity), 4), 256)
    per_row = 4 * ldx + 4 * ld16 + 4 + 4 + 8 + 2 * (4 + 8) + (4 if n_classes else 0) + (8 if weighted else 0)
    return (n * per_row + int(acc_ws_bytes(n, cap, ldx)) + int(bmu_ws_bytes(n, 2))
            + _map_bytes(capacity, ldx, ld16, n_classes, False))


def streamed_bytes(rows: int, n: int, d: int, capacity: int, n_classes: int, weighted: bool,
                   acc_ws_bytes: Callable[[int, int, int], int], bmu_ws_bytes: Callable[[int, int], int]) -> int:
    """Device bytes of a streamed fit with chunks of `rows` rows: the per-sample vectors that stay resident (int32
    winners, the int32 chunk-local sort permutation, labels, weights), two float32 chunk slots, and for one chunk
    the shadows, the post-training winners and distances and the K2 / BMU workspaces; plus the map buffers."""
    ldx, ld16 = _widths(d)
    cap = _round_up(max(int(capacity), 4), 256)
    per_sample = 4 + 4 + (4 if n_classes else 0) + (8 if weighted else 0)
    per_chunk_row = 2 * 4 * ldx + 4 * ld16 + 4 + 2 * (4 + 8)
    return (n * per_sample + rows * per_chunk_row + int(acc_ws_bytes(rows, cap, ldx)) + int(bmu_ws_bytes(rows, 2))
            + _map_bytes(capacity, ldx, ld16, n_classes, True))


def plan_stream(n: int, d: int, capacity: int, n_classes: int, weighted: bool, free_bytes: int,
                acc_ws_bytes: Callable[[int, int, int], int], bmu_ws_bytes: Callable[[int, int], int]) -> int | None:
    """None when the resident fit fits in `free_bytes`, else the chunk row count of a streamed fit: the largest
    multiple of ROW_GRANULE whose footprint fits, at most MAX_CHUNK_BYTES of float32 rows and no more than N
    rounded up.  Raises MemoryError when even two chunks of ROW_GRANULE rows do not fit."""
    n, d = int(n), int(d)
    args = (d, capacity, n_classes, weighted, acc_ws_bytes, bmu_ws_bytes)
    if resident_bytes(n, *args) <= free_bytes:
        return None
    ldx, _ = _widths(d)
    hi = max(1, min(_round_up(max(n, 1), ROW_GRANULE), MAX_CHUNK_BYTES // (4 * ldx)) // ROW_GRANULE)
    if streamed_bytes(ROW_GRANULE, n, *args) > free_bytes:
        fixed = streamed_bytes(ROW_GRANULE, 0, *args)
        per_sample = 4 + 4 + (4 if n_classes else 0) + (8 if weighted else 0)
        raise MemoryError(
            f"{n} samples of {d} features do not fit on the device even when streamed: that needs {per_sample} bytes "
            f"per sample plus {fixed} bytes for the map and two chunks of {ROW_GRANULE} rows, and {int(free_bytes)} "
            f"bytes are free (the resident fit needs {resident_bytes(n, *args)})"
        )
    lo = 1  # fits; find the largest k <= hi with streamed_bytes(k * ROW_GRANULE) <= free_bytes
    while lo < hi:
        mid = (lo + hi + 1) // 2
        if streamed_bytes(mid * ROW_GRANULE, n, *args) <= free_bytes:
            lo = mid
        else:
            hi = mid - 1
    return lo * ROW_GRANULE


def chunk_bounds(n: int, rows: int) -> list[tuple[int, int]]:
    """[c0, c1) row ranges of chunks of `rows` rows; the last one is ragged."""
    return [(c0, min(n, c0 + rows)) for c0 in range(0, n, rows)]


def stream_rows_from_env() -> int:
    """DBGSOM_STREAM_ROWS=n: force streaming with chunks of n rows (rounded up to ROW_GRANULE); 0 / unset = plan."""
    v = int(os.environ.get("DBGSOM_STREAM_ROWS", "0") or 0)
    return _round_up(v, ROW_GRANULE) if v > 0 else 0


class HostStager:
    """A fixed ring of page-locked float32 buffers [RING_PIECES, piece_rows, ldx] between the user's array and the
    device.  Worker threads convert row pieces of the user's array (float32 or float64, any layout, a np.memmap
    included) to float32 in the ring -- float64 rounds to nearest, as the resident upload does -- while the caller
    copies earlier pieces to the device and computes on them.  A buffer is refilled only after the device copy out
    of it has completed (an event the caller hands back).  The padding columns [D, ldx) stay zero.

    The ring is page-locked with cudaHostRegister once and unregistered in `close`; the worker threads live for
    one pass (`pieces`) and are joined when it ends, normally or by an exception."""

    def __init__(self, torch, piece_rows: int, d: int, ldx: int, workers: int | None = None):
        self.torch = torch
        self.d, self.ldx = int(d), int(ldx)
        self.piece_rows = max(1, int(piece_rows))
        self.buf = np.zeros((RING_PIECES, self.piece_rows, self.ldx), dtype=np.float32)
        self.host = torch.from_numpy(self.buf)
        self.workers = workers or max(1, min(RING_PIECES, (os.cpu_count() or 2) // 2))
        self._registered = False
        if self.buf.nbytes:
            torch.cuda.check_error(torch.cuda.cudart().cudaHostRegister(self.buf.ctypes.data, self.buf.nbytes, 0))
            self._registered = True
        self._busy = [None] * RING_PIECES  # event of the last device copy out of each buffer
        self.bytes_staged = 0              # float32 bytes written into the ring
        self.fill_seconds = 0.0            # summed over the workers
        self._lock = threading.Lock()

    @staticmethod
    def piece_rows_for(chunk_rows: int, ldx: int) -> int:
        return max(1, min(int(chunk_rows), RING_PIECE_BYTES // (4 * int(ldx))))

    def close(self) -> None:
        """Unregister the ring.  The caller has synchronised every stream that copies out of it."""
        if self._registered:
            self.torch.cuda.check_error(self.torch.cuda.cudart().cudaHostUnregister(self.buf.ctypes.data))
            self._registered = False
        self._busy = [None] * RING_PIECES
        self.host = self.buf = None

    def _fill(self, slot: int, busy, X, r0: int, r1: int) -> None:
        if busy is not None:
            busy.synchronize()
        t0 = time.perf_counter()
        np.copyto(self.buf[slot, : r1 - r0, : self.d], X[r0:r1], casting="same_kind")
        with self._lock:
            self.fill_seconds += time.perf_counter() - t0
            self.bytes_staged += (r1 - r0) * self.d * 4

    @contextlib.contextmanager
    def pieces(self, X, chunks):
        """Context manager over an iterator of (chunk, r0, r1, host rows [r1 - r0, ldx], release) in row order,
        every piece within one chunk.  The caller enqueues the copy of a piece's rows and calls
        `release(event)` with an event recorded after that copy, before it asks for the next piece."""
        plan = [(c, r0, min(c1, r0 + self.piece_rows)) for c, (c0, c1) in enumerate(chunks)
                for r0 in range(c0, c1, self.piece_rows)]
        pool = ThreadPoolExecutor(max_workers=self.workers, thread_name_prefix="dbgsom-stage")
        pending = collections.deque()

        def submit(k):
            if k < len(plan):
                slot = k % RING_PIECES
                _, r0, r1 = plan[k]
                pending.append(pool.submit(self._fill, slot, self._busy[slot], X, r0, r1))

        def gen():
            for k in range(min(RING_PIECES, len(plan))):
                submit(k)
            for k, (c, r0, r1) in enumerate(plan):
                pending.popleft().result()
                slot = k % RING_PIECES
                released = []

                def release(event, slot=slot, released=released):
                    self._busy[slot] = event
                    released.append(True)

                yield c, r0, r1, self.host[slot, : r1 - r0], release
                if not released:
                    raise RuntimeError("a staged piece was not released")
                submit(k + RING_PIECES)

        try:
            yield gen()
        finally:
            for f in pending:
                f.cancel()
            pool.shutdown(wait=True)
