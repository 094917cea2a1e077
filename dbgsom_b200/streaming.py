"""Fits whose samples do not fit in device memory: chunk planning and the pinned host staging ring.

When the resident fit (every sample, its fp16 shadows and the per-sample buffers of the search, K2 and the
post-training passes in HBM) would not fit in free device memory, `DeviceEngine` keeps only per-sample vectors on
the device and streams the rows from the user's host array in chunks, every epoch.  `plan_stream` decides which of
the two a fit takes and how large the chunks are; `StreamedSamples` is the engine's source of such samples, and
`HostStager` moves the rows through a fixed ring of page-locked buffers.  DESIGN.md, "Streaming fits", describes the
pipeline.
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

from . import _native as nat

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


class StreamedSamples:
    """Samples that stay in the caller's host array (float32 or float64) and pass through the device in chunks of
    `chunk_rows` rows every epoch; the operations of engine.ResidentSamples.  On the device: two float32 chunk slots,
    the fp16 shadows of one chunk, rebuilt for every chunk of every pass, and `row_perm`, the chunk-local order K2
    left each chunk's samples in.  Other chunk buffers are single, because all compute runs on one stream."""

    streaming = True
    winner_cols = 1  # only the int32 winner of every sample stays resident

    def __init__(self, eng, X, rows: int):
        if X.dtype not in (np.float32, np.float64):
            raise ValueError("streamed samples must be float32 or float64")
        torch = eng.torch
        self.eng, self.host_X = eng, X
        n = int(X.shape[0])
        self.chunk_rows = int(min(rows, _round_up(max(n, 1), ROW_GRANULE)))
        self.chunks = chunk_bounds(n, self.chunk_rows)
        self.slots = [torch.empty((self.chunk_rows, eng.ldx), dtype=torch.float32, device=eng.dev) for _ in range(2)]
        self.slot_ready = [torch.cuda.Event() for _ in range(2)]
        self.slot_free = [torch.cuda.Event() for _ in range(2)]
        self.row_perm = torch.empty(n, dtype=torch.int32, device=eng.dev)
        self._chunks_sorted = False  # row_perm holds every chunk's K2 order (after the first epoch)
        self._sorted_search = False  # some chunk's search read its samples sorted (the post passes then do too)
        self._x16 = None
        self.copy_stream = torch.cuda.Stream(eng.dev)
        self.stager = HostStager(torch, HostStager.piece_rows_for(self.chunk_rows, eng.ldx), eng.D, eng.ldx)

    def chunk_pass(self, body) -> None:
        """One pass over the samples in chunks: body(c, c0, c1, x) enqueues the work on chunk c, whose float32 rows
        x [c1 - c0, ldx] are in a device slot.  The rows of chunk c + 1 are staged by the host threads and copied on
        a side stream into the other slot while chunk c is computed; a slot is overwritten only after the work on
        the chunk before has been enqueued and has run (event `slot_free`)."""
        torch = self.eng.torch
        main = torch.cuda.current_stream(self.eng.dev)
        copy = self.copy_stream
        copy.wait_stream(main)  # earlier readers of the slots are done before they are overwritten
        with self.stager.pieces(self.host_X, self.chunks) as pieces:
            pieces = iter(pieces)

            def upload(c):
                s, (c0, c1) = c % 2, self.chunks[c]
                if c >= 2:
                    copy.wait_event(self.slot_free[s])
                done = c0
                with torch.cuda.stream(copy):
                    while done < c1:
                        _, r0, r1, host, release = next(pieces)
                        self.slots[s][r0 - c0 : r1 - c0].copy_(host, non_blocking=True)
                        ev = torch.cuda.Event()
                        ev.record(copy)
                        release(ev)
                        done = r1
                    self.slot_ready[s].record(copy)

            upload(0)
            for c, (c0, c1) in enumerate(self.chunks):
                s = c % 2
                main.wait_event(self.slot_ready[s])
                body(c, c0, c1, self.slots[s][: c1 - c0])
                self.slot_free[s].record(main)
                if c + 1 < len(self.chunks):
                    upload(c + 1)

    def shadows(self, c: int, x, backend, selective):
        """(shadows, row order) for a search of chunk c (rows x) with `backend`; (None, None) for the SIMT search.
        An epoch search (`selective` True or False) reads them sorted by the chunk's K2 order iff it is selective, a
        post-training search (`selective` None) iff some epoch's search was.  D > 256 chunks are never selective, so
        they stay in natural order, where the resident fit keeps them too."""
        if backend[0] != nat.BMU_TENSOR:
            return None, None
        eng, torch = self.eng, self.eng.torch
        need_lo = backend[1] == 3
        self._sorted_search |= bool(selective)
        c0, c1 = self.chunks[c]
        perm = self.row_perm[c0:c1] if (self._sorted_search if selective is None else selective) else None
        if self._x16 is None or (need_lo and self._x16[1] is None):
            self._x16 = (torch.empty((self.chunk_rows, eng.ld16), dtype=torch.float16, device=eng.dev),
                         torch.empty((self.chunk_rows, eng.ld16), dtype=torch.float16, device=eng.dev) if need_lo else None,
                         torch.empty(self.chunk_rows, dtype=torch.float32, device=eng.dev))
        n = c1 - c0
        hi, lo, xn = self._x16[0][:n], (self._x16[1][:n] if need_lo else None), self._x16[2][:n]
        with eng._Phase(eng, "prepare_x16"):
            eng._prepare_x16(x, n, hi, lo, xn, perm)
        return (hi, lo, xn), perm

    def has_order(self, c: int) -> bool:
        return self._chunks_sorted

    def after_k2(self, c: int, order, eligible: bool) -> None:
        """Keep chunk c's K2 order (`order`, chunk-local) for the shadows of its next epoch."""
        c0, c1 = self.chunks[c]
        self.row_perm[c0:c1].copy_(order)
        self._chunks_sorted = True

    def shift_row(self):
        return self.start_rows(np.zeros(1, dtype=np.int64))[0].float()  # float32 -> float64 -> float32 is exact

    def start_rows(self, rows: np.ndarray):
        """float64 [len(rows), ldx] copies of the given local sample rows, rounded through float32 like the chunks."""
        eng = self.eng
        out = np.zeros((len(rows), eng.ldx), dtype=np.float64)
        out[:, : eng.D] = np.asarray(self.host_X[rows]).astype(np.float32)
        return eng.torch.from_numpy(out).to(eng.dev)

    def close(self) -> None:
        if self.stager is not None:
            # no copy may still read the page-locked ring when it is unregistered
            self.eng.torch.cuda.synchronize(self.eng.dev)
            self.stager.close()
            self.stager = None
        self.host_X = self.slots = self.row_perm = self._x16 = None
