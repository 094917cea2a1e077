"""Device engine: owns the HBM buffers of one fit and drives the sm_100a kernels.

PyTorch is used for device memory, streams and (when sharded) `torch.distributed`; every
numeric step is a call into libdbgsom_b200.so through `_native` (include/dbgsom_b200.h).
The engine mirrors the numeric seam of the reference's epoch body
(`dbgsom/BaseSom.py:394-407`): BMU search -> sample weights + per-BMU sums -> neighbourhood
smoothing, with the prototypes resident on the GPU for the whole fit.

There is deliberately no CPU path here: constructing the engine without CUDA raises.
"""

from __future__ import annotations

import math
import os
from typing import Sequence

import numpy as np

from . import _native as nat
from . import streaming
from .hostmath import class_entropy, column_moments_to_stats

_UPLOAD_ROWS = 1 << 20


def scatter_stride(mpad: int) -> int:
    """Stride of the shadow-row permutation: shadow row c holds prototype (c * stride) % mpad.  Close to
    mpad / golden ratio (a low-discrepancy visiting order over the map) and coprime to mpad (a bijection)."""
    stride = int(round(mpad * 0.6180339887498949)) | 1
    while math.gcd(stride, mpad) != 1:
        stride += 2
    return stride


def _round_up(a: int, b: int) -> int:
    return (a + b - 1) // b * b


def map_patch_order(positions: np.ndarray) -> np.ndarray:
    """Prototype indices in Z-order (Morton code) of their grid positions: consecutive runs of 32 / 64 / 128
    prototypes are compact patches of the map (4 x 8, 8 x 8, 8 x 16 cells on a full grid).  The selective BMU search
    lays the shadow columns out in this order, so the prototypes that compete for one sample -- neighbours on the
    map -- share few column tiles."""
    pos = np.asarray(positions, dtype=np.int64).reshape(-1, 2)
    p = pos - pos.min(axis=0)
    code = np.zeros(len(p), dtype=np.int64)
    for b in range(int(max(1, int(p.max()).bit_length()))):
        code |= ((p[:, 0] >> b) & 1) << (2 * b + 1)
        code |= ((p[:, 1] >> b) & 1) << (2 * b)
    return np.argsort(code, kind="stable").astype(np.int32)


class Comm:
    """Thin wrapper over torch.distributed for the single collective of the path."""

    def __init__(self, enabled: bool, device=None):
        self.enabled = bool(enabled)
        self.rank, self.world = 0, 1
        self.device = device  # CUDA device of this rank (object collectives stage through it under NCCL)
        if self.enabled:
            import torch.distributed as dist

            if not dist.is_available() or not dist.is_initialized():
                raise RuntimeError("distributed=True needs an initialised torch.distributed process group")
            self.dist = dist
            self.rank, self.world = dist.get_rank(), dist.get_world_size()

    def allreduce_(self, tensor, op: str = "sum"):
        if self.enabled and self.world > 1:
            ops = {"sum": self.dist.ReduceOp.SUM, "max": self.dist.ReduceOp.MAX, "min": self.dist.ReduceOp.MIN}
            self.dist.all_reduce(tensor, op=ops[op])
        return tensor

    def broadcast_(self, tensor, src: int = 0):
        if self.enabled and self.world > 1:
            self.dist.broadcast(tensor, src=src)
        return tensor

    def _on_device(self):
        import contextlib

        import torch

        if self.device is not None and torch.device(self.device).type == "cuda":
            return torch.cuda.device(self.device)
        return contextlib.nullcontext()

    def broadcast_object(self, obj, src: int = 0):
        """The same Python object on every rank (rank `src`'s).  Used for decisions that must be identical
        everywhere: the start rows drawn from an unseeded generator, for example."""
        if not (self.enabled and self.world > 1):
            return obj
        box = [obj if self.rank == src else None]
        with self._on_device():
            self.dist.broadcast_object_list(box, src=src)
        return box[0]

    def union_sorted(self, values: np.ndarray) -> np.ndarray:
        """Sorted union of the per-rank value sets (class labels of the shards), identical on every rank."""
        if not (self.enabled and self.world > 1):
            return np.asarray(values)
        parts = [None] * self.world
        with self._on_device():
            self.dist.all_gather_object(parts, np.asarray(values))
        return np.unique(np.concatenate([np.asarray(p_) for p_ in parts]))

    def exclusive_offset(self, n_local: int, device) -> tuple[int, int]:
        """(offset of this rank's shard, global sample count)."""
        if not (self.enabled and self.world > 1):
            return 0, n_local
        import torch

        counts = torch.zeros(self.world, dtype=torch.int64, device=device)
        counts[self.rank] = n_local
        self.allreduce_(counts)
        counts = counts.cpu().numpy()
        return int(counts[: self.rank].sum()), int(counts.sum())


class ResidentSamples:
    """Every sample in HBM for the whole fit: X float32 [N, ldx] and its fp16 shadows, which persist between epochs;
    a pass over the samples is one chunk, X itself (streaming.StreamedSamples has the same operations).  Once the
    selective search applies, the shadows are rebuilt in the order K2 grouped the samples by winner (`row_perm`) at
    its first epoch and then every `resort_every` epochs, since each rebuild is a pass over X."""

    streaming = False
    winner_cols = 2  # the epoch winners are [N, 2] (streaming.resident_bytes counts them so)

    def __init__(self, eng, X):
        self.eng, self.X = eng, X
        self.N = int(X.shape[0])
        self.chunks = [(0, self.N)]
        self.X16_hi = self.X16_lo = self.xnorm16 = None
        self.row_perm = None  # int32 [N]: shadow row p holds sample row_perm[p] (None = natural order)
        self.age = 0          # selective-eligible epochs since the shadows were last sorted

    def chunk_pass(self, body) -> None:
        body(0, 0, self.N, self.X)

    def reserve_shadows(self, need_lo: bool) -> bool:
        """Allocate the shadows unless they exist (with the low half when `need_lo`); True when they were allocated,
        in natural order and not yet built."""
        if self.X16_hi is not None and (self.X16_lo is not None or not need_lo):
            return False
        torch, dev, ld16 = self.eng.torch, self.eng.dev, self.eng.ld16
        self.row_perm = None
        self.X16_hi = torch.empty((self.N, ld16), dtype=torch.float16, device=dev)
        self.X16_lo = torch.empty((self.N, ld16), dtype=torch.float16, device=dev) if need_lo else None
        self.xnorm16 = torch.empty(self.N, dtype=torch.float32, device=dev)
        return True

    def shadows(self, c: int, x, backend, selective):
        """(shadows, row order) for a search of chunk c with `backend`; (None, None) for the SIMT search.  Every
        tensor search reads the persistent shadows in their current order, selective (`selective`) or not."""
        if backend[0] != nat.BMU_TENSOR:
            return None, None
        if self.reserve_shadows(backend[1] == 3):
            self.eng._prepare_x16(self.X, self.N, self.X16_hi, self.X16_lo, self.xnorm16)
        return (self.X16_hi, self.X16_lo, self.xnorm16), self.row_perm

    def has_order(self, c: int) -> bool:
        return self.row_perm is not None

    def after_k2(self, c: int, order, eligible: bool) -> None:
        """`order`: K2's winner-sorted permutation of the epoch; `eligible`: the selective search applied to it."""
        if not eligible:
            return
        eng = self.eng
        self.age += 1
        if self.row_perm is None or self.age >= eng.resort_every:
            with eng._Phase(eng, "resort"):
                if self.row_perm is None:
                    self.row_perm = eng.torch.empty(self.N, dtype=eng.torch.int32, device=eng.dev)
                self.row_perm.copy_(order)
                eng._prepare_x16(self.X, self.N, self.X16_hi, self.X16_lo, self.xnorm16, self.row_perm)
            self.age = 0

    def shift_row(self):
        return self.X[0].clone()

    def start_rows(self, rows: np.ndarray):
        """float64 [len(rows), ldx] copies of the given local sample rows."""
        eng, torch = self.eng, self.eng.torch
        src = torch.from_numpy(rows).to(eng.dev)
        out = torch.zeros((len(rows), eng.ldx), dtype=torch.float64, device=eng.dev)
        nat.check(eng.lib.dbgsom_gather_rows(self.X.data_ptr(), eng.ldx, eng.ldx, src.data_ptr(), len(rows),
                                             out.data_ptr(), eng._stream()),
                  "dbgsom_gather_rows")
        eng.launches += 1
        return out

    def close(self) -> None:
        self.X = self.X16_hi = self.X16_lo = self.xnorm16 = self.row_perm = None


def _sample_buffer(name: str):
    """Engine attribute read from the sample source: the resident X, its shadows, the shadow-row order (None where
    the source has no such buffer)."""
    return property(lambda self: getattr(self.samples, name, None))


class DeviceEngine:
    """One fit's worth of device state.  See module docstring."""

    X, X16_hi, X16_lo, xnorm16, row_perm = map(_sample_buffer, ("X", "X16_hi", "X16_lo", "xnorm16", "row_perm"))

    # M^2 D above which the smoothing rows are split over the ranks (DBGSOM_K3_SHARD_MIN_WORK overrides; tests)
    K3_SHARD_MIN_WORK = int(os.environ.get("DBGSOM_K3_SHARD_MIN_WORK", 1 << 36))

    def __init__(
        self,
        device: str = "cuda",
        bmu_backend: str = "auto",
        distributed: bool = False,
        bound_scale: float = 0.0,
        strict_ties: bool = False,
        capacity_hint: int = 0,
    ) -> None:
        import torch

        self.torch = torch
        self.lib = nat.load()
        if not torch.cuda.is_available():
            raise RuntimeError("dbgsom_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.dev = torch.device(device)
        if self.dev.type != "cuda":
            raise ValueError(f"device must be a CUDA device, got {device!r}")
        if self.dev.index is None:
            self.dev = torch.device("cuda", torch.cuda.current_device())
        nat.check(self.lib.dbgsom_check_device(self.dev.index), "dbgsom_check_device")
        if bmu_backend not in ("auto", "tensor", "tensor1", "simt"):
            raise ValueError("bmu_backend must be 'auto', 'tensor', 'tensor1' or 'simt'")
        self.bmu_backend = bmu_backend
        self.bound_scale = float(bound_scale)
        self.strict_ties = bool(strict_ties)
        # Selective search (csrc/bmu_tc.cu, SEL): one fp16 pass over everything, split-fp16 passes only over the
        # column tiles it cannot rule out.  Needs the samples sorted by winner (rebuilt every `resort_every` epochs
        # from the permutation K2 leaves behind) and the shadow columns in map-patch order.  DBGSOM_SELECT=0 turns it off.
        self.select_enabled = os.environ.get("DBGSOM_SELECT", "1") != "0"
        self.select_granule = int(os.environ.get("DBGSOM_SELECT_GRANULE", "64"))
        # Per-tile error bounds for the streamed search (D > 256, one winner; csrc/bmu_tc.cu, TB): the rounding bound of a
        # score follows the norms of the prototypes of ITS column tile, which are coherent when the shadow columns are
        # laid out in map patches.  DBGSOM_TILE_BOUND=0 turns it off (map-wide maxima everywhere, scattered columns).
        self.tile_bounds_enabled = os.environ.get("DBGSOM_TILE_BOUND", "1") != "0"
        self.tile_bound = None
        self._tile_ready = False
        self.resort_every = int(os.environ.get("DBGSOM_RESORT_EVERY", "8"))
        self.tile_mask = None
        self._map_order = None    # prototype indices in map-patch order (from the topology)
        self._perm_cache = {}
        self._epoch_kinds = {"selective": 0, "classic": 0}
        self.comm = Comm(distributed, self.dev)
        self.sample_offset = 0
        self.n_samples_global = 0
        self.weight = None        # float64 [N] frequency weights of the samples (None: unweighted)
        self.weight_total = 0.0   # sum of the weights over all ranks (== n_samples_global when unweighted)
        self.launches = 0  # kernels + memsets enqueued by this engine (bench bookkeeping)
        self.fp32_reruns = 0  # epochs repeated on the fp32 search because a prototype left the fp16 range
        self._prof = None
        self.last_bmu_stats = None
        self._ws = {}
        self.samples = None       # ResidentSamples or streaming.StreamedSamples: where the fit's samples live
        self.W = None
        self.M = 0
        self.n_previous_rows = 0
        # Streaming (streaming.py, DESIGN.md "Streaming fits"): samples that do not fit in device memory stay in the
        # caller's host array and pass through the device in chunks of `stream_rows` rows every epoch.  0 plans
        # automatically (stream only when the resident fit would not fit); DBGSOM_STREAM_ROWS=n forces chunks of n rows.
        self.stream_rows = streaming.stream_rows_from_env()
        self.capacity_hint = int(capacity_hint)  # map capacity the fit will ask for (sizes the plan)
        self._copy_stream = None  # side stream of `epoch_from_host`

    @property
    def streaming(self) -> bool:
        """The samples stay in host memory and pass through the device in chunks every epoch."""
        return self.samples is not None and self.samples.streaming

    @property
    def chunks(self):
        """[(c0, c1)] row ranges of one pass over the samples ([(0, N)] when resident)."""
        return None if self.samples is None else self.samples.chunks

    @property
    def chunk_rows(self) -> int:
        return self.samples.chunk_rows

    # ------------------------------------------------------------------ helpers
    def _stream(self):
        return self.torch.cuda.current_stream(self.dev).cuda_stream

    def enable_profiling(self, on: bool = True) -> None:
        """Record CUDA-event pairs around every phase of `epoch` (read with `phase_times_ms`)."""
        self._prof = {} if on else None

    class _Phase:
        def __init__(self, eng, name):
            self.eng, self.name = eng, name

        def __enter__(self):
            if self.eng._prof is not None:
                ev = self.eng.torch.cuda.Event
                self.t0, self.t1 = ev(enable_timing=True), ev(enable_timing=True)
                self.t0.record(self.eng.torch.cuda.current_stream(self.eng.dev))

        def __exit__(self, *exc):
            if self.eng._prof is not None:
                self.t1.record(self.eng.torch.cuda.current_stream(self.eng.dev))
                self.eng._prof.setdefault(self.name, []).append((self.t0, self.t1))

    def phase_times_ms(self, reset: bool = True) -> dict:
        """Mean device time per phase and call over the recorded epochs (synchronises)."""
        self.torch.cuda.synchronize(self.dev)
        out = {k: [a.elapsed_time(b) for a, b in v] for k, v in (self._prof or {}).items()}
        if reset and self._prof is not None:
            self._prof = {}
        return out

    def _workspace(self, key: str, nbytes: int):
        buf = self._ws.get(key)
        if buf is None or buf.numel() < nbytes:
            buf = self.torch.empty(max(int(nbytes), 256), dtype=self.torch.uint8, device=self.dev)
            self._ws[key] = buf
        return buf

    def _upload_matrix(self, X: np.ndarray):
        """Host [N, D] (float32/float64) -> device float32 [N, ldx], zero padded to ldx = 4k."""
        torch = self.torch
        n, d = X.shape
        ldx = _round_up(d, 4)
        out = torch.zeros((n, ldx), dtype=torch.float32, device=self.dev) if ldx != d else torch.empty(
            (n, ldx), dtype=torch.float32, device=self.dev
        )
        for s in range(0, n, _UPLOAD_ROWS):
            chunk = np.ascontiguousarray(X[s : s + _UPLOAD_ROWS])
            out[s : s + chunk.shape[0], :d] = torch.from_numpy(chunk).to(self.dev, non_blocking=False).to(torch.float32)
        return out

    def close(self) -> None:
        if self.samples is not None:
            self.samples.close()
        self._ws.clear()
        self._perm_cache.clear()
        for name in ("W", "W32", "W16_hi", "W16_lo", "Wb16", "_row_hash", "labels", "weight", "part", "hop", "_final_idx",
                     "tile_mask", "tile_bound", "_cpart", "_chist"):
            if hasattr(self, name):
                setattr(self, name, None)

    # ------------------------------------------------------------------ data
    def load_data(self, X: np.ndarray, y, n_classes: int, sample_weight=None) -> dict:
        """Upload the samples and reduce the column statistics `fit` needs (K4).  Samples that would not fit in
        device memory (or `stream_rows` > 0) stay in X and are streamed in chunks every epoch.

        `sample_weight` (float64 [N], finite, >= 0; this rank's shard): frequency weights -- a sample of weight w
        counts like w copies of it in every sum of the fit.  None runs the unweighted kernels."""
        torch = self.torch
        with torch.cuda.device(self.dev):
            self.N, self.D = int(X.shape[0]), int(X.shape[1])
            self.ldx = _round_up(self.D, 4)
            rows = self._plan_rows(self.N, self.D, int(n_classes) if y is not None else 0, sample_weight is not None)
            samples = ResidentSamples(self, self._upload_matrix(X)) if rows is None else streaming.StreamedSamples(
                self, X, rows)
            labels = None if y is None else torch.from_numpy(np.ascontiguousarray(y, dtype=np.int32)).to(self.dev)
            weight = None if sample_weight is None else torch.from_numpy(
                np.ascontiguousarray(sample_weight, dtype=np.float64)).to(self.dev)
            return self._use_samples(samples, labels, n_classes, weight)

    def _use_samples(self, samples, labels, n_classes: int, weight) -> dict:
        self.samples = samples
        self.ld16 = _round_up(self.ldx, 64)
        self.n_classes, self.labels = int(n_classes), labels
        self.sample_offset, self.n_samples_global = self.comm.exclusive_offset(self.N, self.dev)
        self._set_weights(weight)
        self.idx = self.torch.empty((self.N, samples.winner_cols), dtype=self.torch.int32, device=self.dev)
        return self._column_statistics()

    def free_device_bytes(self) -> int:
        """Device bytes a fit may still allocate: free memory plus what torch has cached but not handed out, less
        `streaming.free_margin`."""
        free, total = self.torch.cuda.mem_get_info(self.dev)
        cached = self.torch.cuda.memory_reserved(self.dev) - self.torch.cuda.memory_allocated(self.dev)
        return int(free) + int(cached) - streaming.free_margin(total)

    def _plan_rows(self, n: int, d: int, n_classes: int, weighted: bool, capacity: int | None = None) -> int | None:
        """Chunk rows of a streamed fit, or None for the resident one (`streaming.plan_stream`)."""
        if self.stream_rows > 0:
            return streaming._round_up(int(self.stream_rows), streaming.ROW_GRANULE)
        cap = max(int(self.capacity_hint if capacity is None else capacity), 4)
        return streaming.plan_stream(n, d, cap, n_classes, weighted, self.free_device_bytes(),
                                     self.lib.dbgsom_accumulate_workspace_bytes, self.lib.dbgsom_bmu_workspace_bytes)

    def _set_weights(self, weight_dev) -> None:
        self.weight = weight_dev
        if weight_dev is None:
            self.weight_total = float(self.n_samples_global)
            return
        if weight_dev.dtype != self.torch.float64 or tuple(weight_dev.shape) != (self.N,) or not weight_dev.is_contiguous():
            raise ValueError("sample_weight must be a contiguous float64 vector with one entry per sample")
        total = weight_dev.sum().reshape(1)
        self.weight_total = float(self.comm.allreduce_(total).item())

    def _colstats_parts(self, X, n: int, shift_row, weight) -> np.ndarray:
        """K4 over n rows of X: the [COLSTATS_PARTS, 2 ldx + 1] row-block parts on the host."""
        parts = self.torch.zeros((nat.COLSTATS_PARTS, 2 * self.ldx + 1), dtype=self.torch.float64, device=self.dev)
        if weight is None:
            nat.check(
                self.lib.dbgsom_colstats(
                    X.data_ptr(), n, self.ldx, self.ldx, shift_row.data_ptr(), parts.data_ptr(), self._stream()
                ),
                "dbgsom_colstats",
            )
        else:
            nat.check(
                self.lib.dbgsom_colstats_weighted(
                    X.data_ptr(), n, self.ldx, self.ldx, shift_row.data_ptr(), weight.data_ptr(),
                    parts.data_ptr(), self._stream(),
                ),
                "dbgsom_colstats_weighted",
            )
        self.launches += 1
        return parts.cpu().numpy()

    def _column_statistics(self) -> dict:
        torch = self.torch
        # K4: moments about a common data row (rank 0's first row, as float32)
        shift_row = self.samples.shift_row()
        self.comm.broadcast_(shift_row, 0)
        # the row-block parts of a chunk are added on the host, then the chunk sums in chunk order: the same
        # statistics on every run
        acc = []

        def body(c, c0, c1, x):
            p = self._colstats_parts(x, c1 - c0, shift_row, self.weight[c0:c1] if self.weight is not None else None)
            sums, maxabs = p[:, : 2 * self.ldx].sum(axis=0), p[:, 2 * self.ldx].max()
            acc[:] = [sums, maxabs] if c == 0 else [acc[0] + sums, max(acc[1], maxabs)]

        self.samples.chunk_pass(body)
        moments = torch.from_numpy(np.append(*acc)).to(self.dev)
        self.comm.allreduce_(moments[: 2 * self.ldx])
        self.comm.allreduce_(moments[2 * self.ldx :], "max")
        m = moments.cpu().numpy()
        s1, s2, maxabs = m[: self.ldx], m[self.ldx : 2 * self.ldx], float(m[2 * self.ldx])
        # the amount of data is the total weight (the sample count when unweighted)
        n_g = self.weight_total if self.weight is not None else self.n_samples_global
        stats = column_moments_to_stats(n_g, s1, s2)
        stats["n_samples"] = int(self.n_samples_global)
        if self.weight is not None:
            stats["total_weight"] = n_g
        self.total_variance = stats["total_variance"]
        # data mean (centres the fp16 shadow) and a power-of-two scale that keeps it in range
        mean = shift_row.double().cpu().numpy() + s1 / n_g
        # the device copy of X is float32: an offset far larger than the spread costs that many digits of the spread
        std = np.sqrt(np.maximum(s2 - s1 * s1 / n_g, 0.0) / max(n_g, 1))
        with np.errstate(divide="ignore", invalid="ignore"):
            ratio = np.where(std > 0, np.abs(mean) / std, 0.0)
        if ratio.size and float(ratio.max()) > 1e3:
            import warnings

            warnings.warn(
                f"column {int(ratio.argmax())} has |mean| / std = {float(ratio.max()):.3g}: samples are stored as float32 on the "
                "device, so about that many digits of the column's spread are lost; centre the data before fitting",
                RuntimeWarning, stacklevel=3,
            )
        self.shift = torch.from_numpy(mean.astype(np.float32)).to(self.dev)
        # |x'| <= 2^12 leaves a factor 16 of fp16 range for prototypes outside the data hull
        self.scale = 1.0 if not (maxabs > 0 and math.isfinite(maxabs)) else 2.0 ** math.floor(
            math.log2(2.0**12 / (2.0 * maxabs))
        )
        return stats

    def load_device_data(self, X_dev, labels_dev=None, n_classes: int = 0, weight_dev=None) -> dict:
        """Like `load_data` for samples that already live in HBM (float32 [N, D], D % 4 == 0; weights float64 [N])."""
        torch = self.torch
        if X_dev.dtype != torch.float32 or X_dev.dim() != 2 or not X_dev.is_contiguous() or X_dev.shape[1] % 4:
            raise ValueError("X_dev must be a contiguous float32 [N, D] CUDA tensor with D % 4 == 0")
        with torch.cuda.device(self.dev):
            self.N, self.D = int(X_dev.shape[0]), int(X_dev.shape[1])
            self.ldx = self.D
            return self._use_samples(ResidentSamples(self, X_dev), labels_dev, n_classes, weight_dev)

    def _prepare_x16(self, x, n: int, hi, lo, xnorm, perm=None) -> None:
        """fp16 shadows hi (and lo, when given) and xnorm of n rows of x, in the order `perm` when given."""
        lo_ptr = lo.data_ptr() if lo is not None else None
        if perm is None:
            nat.check(self.lib.dbgsom_prepare_x16(x.data_ptr(), n, self.ldx, self.ldx, self.shift.data_ptr(), self.scale,
                                                  hi.data_ptr(), lo_ptr, self.ld16, xnorm.data_ptr(), self._stream()),
                      "dbgsom_prepare_x16")
            self.launches += 1
        else:
            nat.check(self.lib.dbgsom_prepare_x16_sorted(x.data_ptr(), n, self.ldx, self.ldx, self.shift.data_ptr(),
                                                         self.scale, perm.data_ptr(), hi.data_ptr(), lo_ptr, self.ld16,
                                                         xnorm.data_ptr(), self._stream()),
                      "dbgsom_prepare_x16_sorted")
            self.launches += 2

    # ------------------------------------------------------------------ map state
    def _alloc_map(self, capacity: int) -> None:
        torch = self.torch
        cap = _round_up(max(int(capacity), 4), 256)
        old = self.W
        self.cap = cap
        self.W = [torch.zeros((cap, self.ldx), dtype=torch.float64, device=self.dev) for _ in range(2)]
        self.W32 = torch.zeros((cap, self.ldx), dtype=torch.float32, device=self.dev)
        self.W16_hi = self.W16_lo = None
        self.wnorm = torch.empty(cap, dtype=torch.float32, device=self.dev)
        self.wshift = torch.empty(self.ldx, dtype=torch.float64, device=self.dev)
        self.wmax = torch.zeros(4, dtype=torch.float32, device=self.dev)  # see dbgsom_prepare_w
        self.part = torch.zeros(cap * self.ldx + 3 * cap, dtype=torch.float64, device=self.dev)
        self.change = torch.zeros(1, dtype=torch.float64, device=self.dev)
        self.bmu_stats = torch.zeros(8, dtype=torch.int64, device=self.dev)
        # weighted fits sum the class histogram as float64 weights
        hist_dtype = torch.int32 if self.weight is None else torch.float64
        self.class_hist = (
            torch.zeros((cap, self.n_classes), dtype=hist_dtype, device=self.dev) if self.labels is not None else None
        )
        if self.samples is not None and len(self.samples.chunks) > 1:
            # one chunk's K2 sums and class histogram, added into the epoch's in chunk order
            self._cpart = torch.empty_like(self.part)
            self._chist = torch.empty_like(self.class_hist) if self.class_hist is not None else None
        if old is not None:
            for new, prev in zip(self.W, old):
                new[: prev.shape[0]] = prev

    def _ensure_capacity(self, m: int) -> None:
        if m > self.cap:
            self._alloc_map(max(2 * self.cap, m))

    def init_map_from_rows(self, rows: Sequence[int], capacity: int) -> None:
        """Start prototypes = the given global sample rows (dbgsom/BaseSom.py:423-430)."""
        torch = self.torch
        with torch.cuda.device(self.dev):
            self.W = None
            self._alloc_map(capacity)
            self.cur = 0
            rows = np.asarray(rows, dtype=np.int64)
            local = rows - self.sample_offset
            owned = (local >= 0) & (local < self.N)
            W0 = self.W[0]
            if owned.any():
                tmp = self.samples.start_rows(np.where(owned, local, 0))
                tmp[torch.from_numpy(~owned).to(self.dev)] = 0
                W0[: len(rows)] = tmp
            else:
                W0[: len(rows)] = 0
            self.comm.allreduce_(W0[: len(rows)])
            self.M = len(rows)
            self.n_previous_rows = self.M

    def set_map(self, W: np.ndarray) -> None:
        """Replace the prototypes by a host matrix [M, D] (fixed-map training, tests)."""
        torch = self.torch
        with torch.cuda.device(self.dev):
            m = int(W.shape[0])
            if self.W is None:
                self._alloc_map(m)
                self.cur = 0
            self._ensure_capacity(m)
            cur = self.W[self.cur]
            cur.zero_()
            cur[:m, : self.D] = torch.from_numpy(np.ascontiguousarray(W, dtype=np.float64)).to(self.dev)
            self.M = m
            self.n_previous_rows = m

    def set_hops(self, hop_u16: np.ndarray, positions: np.ndarray | None = None) -> None:
        torch = self.torch
        m = hop_u16.shape[0]
        self._map_order = map_patch_order(positions) if positions is not None else None
        finite = hop_u16[hop_u16 != 0xFFFF]
        self.hop_max = int(finite.max()) if finite.size else 0
        # uint16 travels as int16 bit patterns (torch has no uint16 arithmetic; none is needed)
        self.hop = torch.from_numpy(np.ascontiguousarray(hop_u16).view(np.int16)).to(self.dev)
        self.ldh = m

    def set_hops_from_topology(self, topo) -> None:
        """All-pairs hop counts of the map graph, computed on the device (one BFS per source node,
        `dbgsom_hops`) from the adjacency table; only maps beyond the kernel's shared-memory limit
        take the host BFS of `MapTopology.hop_matrix_u16`.  Replaces the per-epoch
        `nx.floyd_warshall_numpy` of dbgsom/BaseSom.py:401."""
        torch = self.torch
        m = len(topo)
        if m > nat.HOPS_MAX_M:
            self.set_hops(topo.hop_matrix_u16(), topo.positions())
            return
        self._map_order = map_patch_order(topo.positions())
        with torch.cuda.device(self.dev):
            d_adj = torch.from_numpy(topo.adjacency_table()).to(self.dev)
            self.hop = torch.empty((m, m), dtype=torch.int16, device=self.dev)
            nat.check(self.lib.dbgsom_hops(d_adj.data_ptr(), m, self.hop.data_ptr(), m, self._stream()), "dbgsom_hops")
            self.launches += 1
            self.ldh = m
            # 0xFFFF (unreachable) reads as -1 in the int16 view, so the maximum is the largest finite hop count
            self.hop_max = max(int(self.hop.max().item()), 0)

    def hops_host(self) -> np.ndarray:
        """The device hop matrix as uint16 on the host (tests)."""
        return self.hop.cpu().numpy().view(np.uint16)

    def apply_row_ops(self, ops, n_rows: int) -> None:
        """Prototype rows of the neurons a growth step inserted (see topology.RowOp)."""
        torch = self.torch
        with torch.cuda.device(self.dev):
            self._ensure_capacity(n_rows)
            flat = np.array([(o.dst, o.a, o.b, o.c) for o in ops], dtype=np.int32).reshape(-1, 4)
            d_ops = torch.from_numpy(flat).to(self.dev)
            nat.check(
                self.lib.dbgsom_apply_row_ops(
                    self.W[self.cur].data_ptr(), self.ldx, d_ops.data_ptr(), len(ops), self._stream()
                ),
                "dbgsom_apply_row_ops",
            )
            self.launches += 1
            self.M = int(n_rows)

    def keep_rows(self, alive: np.ndarray) -> None:
        """Drop all prototype rows but `alive` (dead-neuron removal at the end of fit)."""
        torch = self.torch
        idx = torch.from_numpy(np.asarray(alive, dtype=np.int64)).to(self.dev)
        cur = self.W[self.cur]
        kept = cur.index_select(0, idx)
        cur.zero_()
        cur[: kept.shape[0]] = kept
        self.M = int(kept.shape[0])

    def weights(self) -> np.ndarray:
        return self.W[self.cur][: self.M, : self.D].cpu().numpy()

    # ------------------------------------------------------------------ kernels
    def _pick_backend(self, n: int, m: int) -> tuple[int, int]:
        """(backend, n_pass).  The tensor path pays off once the distance matrix is large."""
        mode = self.bmu_backend
        if mode == "simt":
            return nat.BMU_SIMT, 0
        if mode == "tensor":
            return nat.BMU_TENSOR, 3
        if mode == "tensor1":
            return nat.BMU_TENSOR, 1
        big = m >= 128 and n * m * self.ldx >= (1 << 31)
        return (nat.BMU_TENSOR, 3) if big else (nat.BMU_SIMT, 0)

    def _column_order(self, m: int, mpad: int, map_order: bool):
        """(proto_of_col, col_of_proto, stride) device tables of the shadow-column permutation.

        Classic search: a fixed scattered visiting order (shadow row c holds prototype (c * stride) % mpad, stride ~
        mpad / golden ratio and coprime to mpad) -- a low-discrepancy sequence over the map that the kernel can
        evaluate in registers, so running minima are rarely improved.  Selective search: map-patch order
        (`map_patch_order`), padding columns last."""
        torch = self.torch
        key = (mpad, "map", id(self._map_order)) if map_order else (mpad, "scatter")
        hit = self._perm_cache.get(key)
        if hit is not None:
            return hit
        if map_order:
            stride = 0
            proto_of_col = np.arange(mpad, dtype=np.int32)
            proto_of_col[:m] = self._map_order
        else:
            stride = scatter_stride(mpad)
            proto_of_col = ((np.arange(mpad, dtype=np.int64) * stride) % mpad).astype(np.int32)
            if mpad > 65535:
                stride = 0
            if os.environ.get("DBGSOM_PERM") == "random":  # tuning switch
                proto_of_col = np.random.default_rng(0x5EED + mpad).permutation(mpad).astype(np.int32)
                stride = 0
            if os.environ.get("DBGSOM_PERM") == "table":
                stride = 0
        col_of_proto = np.empty_like(proto_of_col)
        col_of_proto[proto_of_col] = np.arange(mpad, dtype=np.int32)
        hit = (torch.from_numpy(proto_of_col).to(self.dev), torch.from_numpy(col_of_proto).to(self.dev), stride)
        if len(self._perm_cache) > 8:
            self._perm_cache.clear()
        self._perm_cache[key] = hit
        return hit

    def _prepare_w(self, W, m: int, tensor: bool, need_lo: bool, top1: bool = True, map_order: bool = False) -> int:
        torch = self.torch
        mpad = _round_up(m, 256)
        # streamed three-pass search for one winner: per-tile bounds, columns in map patches when a topology is known
        tile = bool(tensor and need_lo and top1 and self.tile_bounds_enabled and self.ld16 > 256)
        if tile and self._map_order is not None and len(self._map_order) == m:
            map_order = True
        self._tile_ready = False
        if tensor:
            self.proto_of_col, self.col_of_proto, self.proto_stride = self._column_order(m, mpad, map_order)
            if self.W16_hi is None or self.W16_hi.shape[0] < mpad or (need_lo and self.W16_lo is None):
                rows = _round_up(max(mpad, self.cap), 256)
                self.W16_hi = torch.zeros((rows, self.ld16), dtype=torch.float16, device=self.dev)
                self.W16_lo = torch.zeros((rows, self.ld16), dtype=torch.float16, device=self.dev) if need_lo else None
                self.wnorm = torch.empty(rows, dtype=torch.float32, device=self.dev)
                # wnorm as an MMA operand (dbgsom_prepare_bias): three fp16 pieces per shadow row, rest stays zero
                self.Wb16 = torch.zeros((rows, 64), dtype=torch.float16, device=self.dev)
                self.bias_scale = torch.zeros(1, dtype=torch.float32, device=self.dev)
        nat.check(
            self.lib.dbgsom_prepare_w(
                W.data_ptr(), m, self.ldx, self.shift.data_ptr(), self.scale, self.W32.data_ptr(),
                self.W16_hi.data_ptr() if tensor else None,
                self.W16_lo.data_ptr() if (tensor and need_lo) else None,
                self.ld16, mpad, self.col_of_proto.data_ptr() if tensor else None,
                self.wnorm.data_ptr() if tensor else None,
                self.wshift.data_ptr() if tensor else None, self.wmax.data_ptr(), self._stream(),
            ),
            "dbgsom_prepare_w",
        )
        self.launches += 3 if tensor else 2
        # top-1 searches: exact copies of a lower-indexed prototype can never win (lowest index takes exact
        # ties), so they leave the candidate search and the epilogue need not order equal scores
        self._ties_any = bool(tensor and top1)
        if self._ties_any:
            if getattr(self, "_row_hash", None) is None or self._row_hash.numel() < m:
                self._row_hash = torch.empty(max(m, self.cap), dtype=torch.int64, device=self.dev)
            nat.check(
                self.lib.dbgsom_exclude_duplicates(
                    W.data_ptr(), m, self.ldx, self.col_of_proto.data_ptr(), self.wnorm.data_ptr(),
                    self._row_hash.data_ptr(), self._stream(),
                ),
                "dbgsom_exclude_duplicates",
            )
            self.launches += 2
        if tile:
            if self.tile_bound is None or self.tile_bound.numel() < mpad // 64:
                self.tile_bound = torch.zeros(_round_up(max(mpad, self.cap), 256) // 64, dtype=torch.float32, device=self.dev)
            nat.check(
                self.lib.dbgsom_tile_bounds(W.data_ptr(), m, self.ldx, self.wshift.data_ptr(), self.scale,
                                            self.proto_of_col.data_ptr(), self.wnorm.data_ptr(), mpad,
                                            self.tile_bound.data_ptr(), self._stream()),
                "dbgsom_tile_bounds",
            )
            self.launches += 1
            self._tile_ready = True
        # experiment, off by default: wnorm enters the accumulator through an extra k-step (dbgsom_prepare_bias).  It
        # halves the epilogue's shared-memory loads but measured no gain (D = 256: MMA bound; D = 128: the epilogue is
        # bound by its instruction count, not by the shared-memory pipe) -- see DESIGN.md, K1.
        # DBGSOM_FLAG_BIAS=1 (off by default) uses it in the FLAG pass of the selective search for D <= 128, whose lean
        # epilogue then needs no per-column load and no FFMA: 12.5M x 128 rows 11.83 -> 11.36 ms (the pass becomes MMA
        # bound including the extra k-step), epoch 21.0 -> 20.7 ms; winners unchanged (c4-shape trajectory test)
        flag_bias = bool(tensor and need_lo and top1 and map_order and not tile and self.ld16 <= 128
                         and os.environ.get("DBGSOM_FLAG_BIAS", "0") == "1")
        self._flag_bias_ready = False
        if flag_bias or (tensor and need_lo and os.environ.get("DBGSOM_TC_BIAS", "0") == "1"):
            nat.check(
                self.lib.dbgsom_prepare_bias(self.wnorm.data_ptr(), mpad, self.wmax.data_ptr(), self.Wb16.data_ptr(),
                                             self.bias_scale.data_ptr(), self._stream()),
                "dbgsom_prepare_bias",
            )
            self.launches += 1
            self._bias_ready = os.environ.get("DBGSOM_TC_BIAS", "0") == "1"
            self._flag_bias_ready = flag_bias
        else:
            self._bias_ready = False
        return mpad

    def _run_bmu(self, X, n: int, ldx: int, x16, W, m: int, n_bmu: int, want_dist: bool, idx, dist, backend=None,
                 strict=None, row_perm=None, selective=False):
        """prepare_w + candidate search + exact re-score for samples X against prototypes W."""
        backend = self._pick_backend(n, m) if backend is None else backend
        mpad = self._prepare_search(W, m, backend, n_bmu, map_order=selective)
        self._bmu_search(X, n, ldx, x16, W, m, mpad, n_bmu, want_dist, idx, dist, backend, strict=strict,
                         row_perm=row_perm, selective=selective)

    def _prepare_search(self, W, m: int, backend, n_bmu: int, map_order: bool = False) -> int:
        """prepare_w for searches of `backend` against the first m rows of W; returns mpad."""
        if W.shape[0] > self.W32.shape[0]:
            self.W32 = self.torch.zeros((W.shape[0], self.ldx), dtype=self.torch.float32, device=self.dev)
        with self._Phase(self, "prepare_w"):
            return self._prepare_w(W, m, backend[0] == nat.BMU_TENSOR, backend[1] == 3, top1=n_bmu == 1,
                                   map_order=map_order)

    def _select_eligible(self, n: int, m: int, backend) -> bool:
        """The selective search applies: tensor search with three passes, one winner, shapes the kernels cover, and a
        topology to order the shadow columns by."""
        if not self.select_enabled or backend != (nat.BMU_TENSOR, 3):
            return False
        if self._map_order is None or len(self._map_order) != m:
            return False
        if _round_up(m, 256) < 1024:  # a handful of column tiles: nothing to select from
            return False
        return bool(self.lib.dbgsom_bmu_select_supported(n, self.ld16, _round_up(m, 256), 1, self.select_granule))

    def _bmu_search(self, X, n, ldx, x16, W, m, mpad, n_bmu, want_dist, idx, dist, backend, ws_key="bmu", strict=None,
                    row_perm=None, selective=False):
        """Candidate search + exact re-score of n sample rows (shadows of W must be current).

        `row_perm`: the shadows are in sorted sample order.  `selective`: FLAG pass (one fp16 pass, which column tiles
        can hold the winner of which row-tile pair) + REFINE pass (three passes over those tiles) instead of the
        classic three passes over everything; needs row_perm and the map-patch column order."""
        be, n_pass = backend
        tensor = be == nat.BMU_TENSOR
        ws_bytes = self.lib.dbgsom_bmu_workspace_bytes(n, n_bmu)
        ws = self._workspace(ws_key, ws_bytes)
        a = nat.BmuArgs()
        a.d_X, a.N, a.D, a.ldx, a.ld16 = X.data_ptr(), n, self.ldx, ldx, self.ld16
        if tensor:
            xh, xl, xn = x16
            a.d_X16_hi, a.d_X16_lo, a.d_xnorm16 = xh.data_ptr(), (xl.data_ptr() if xl is not None else None), xn.data_ptr()
            a.d_W16_hi = self.W16_hi.data_ptr()
            a.d_W16_lo = self.W16_lo.data_ptr() if self.W16_lo is not None else None
            a.d_wnorm = self.wnorm.data_ptr()
            if getattr(self, "_bias_ready", False):
                a.d_Wb16, a.d_bias_scale = self.Wb16.data_ptr(), self.bias_scale.data_ptr()
            a.d_proto_of_col = self.proto_of_col.data_ptr()
            a.proto_stride = self.proto_stride
            a.ties_any = int(self._ties_any and n_bmu == 1)
            if self._tile_ready and n_bmu == 1 and n_pass == 3 and not selective:
                a.d_tile_bound = self.tile_bound.data_ptr()
        a.d_W, a.d_W32, a.d_wmax = W.data_ptr(), self.W32.data_ptr(), self.wmax.data_ptr()
        a.scale, a.M, a.Mpad, a.n_bmu = self.scale, m, mpad, n_bmu
        a.backend, a.n_pass, a.bound_scale, a.tie_rel = be, n_pass, self.bound_scale, 0.0
        a.strict, a.want_dist = int(self.strict_ties if strict is None else strict), int(want_dist)
        a.d_idx, a.d_dist = idx.data_ptr(), (dist.data_ptr() if dist is not None else None)
        a.d_stats = self.bmu_stats.data_ptr()
        a.d_workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
        if tensor and row_perm is not None:
            a.d_row_perm = row_perm.data_ptr()
        if selective:
            n_pairs = -(-(-(-n // 128)) // 2)
            if self.tile_mask is None or self.tile_mask.numel() < n_pairs:
                self.tile_mask = self.torch.zeros(n_pairs, dtype=self.torch.int64, device=self.dev)
            self.tile_mask.zero_()
            a.d_tile_mask = self.tile_mask.data_ptr()
            a.select_granule = self.select_granule
            a.select, a.n_pass = nat.SELECT_FLAG, 1
            if getattr(self, "_flag_bias_ready", False):
                a.d_Wb16, a.d_bias_scale = self.Wb16.data_ptr(), self.bias_scale.data_ptr()
            with self._Phase(self, "bmu_candidates"):
                nat.check(self.lib.dbgsom_bmu_candidates(a, self._stream()), "dbgsom_bmu_candidates[flag]")
            a.d_Wb16, a.d_bias_scale = None, None
            a.select, a.n_pass = nat.SELECT_REFINE, 3
            with self._Phase(self, "bmu_second_stage"):
                nat.check(self.lib.dbgsom_bmu_candidates(a, self._stream()), "dbgsom_bmu_candidates[refine]")
            self.launches += 2
            self._epoch_kinds["selective"] += 1
        else:
            if tensor and n_pass == 3 and n_bmu == 1:
                self._epoch_kinds["classic"] += 1
            with self._Phase(self, "bmu_candidates"):
                nat.check(self.lib.dbgsom_bmu_candidates(a, self._stream()), "dbgsom_bmu_candidates")
        with self._Phase(self, "bmu_resolve"):
            nat.check(self.lib.dbgsom_bmu_resolve(a, self._stream()), "dbgsom_bmu_resolve")
        self.launches += 4  # candidate kernel, queue memset, re-score kernel, re-scan kernel
        self.last_backend = (be, n_pass)

    def epoch_from_host(self, host_X, sigma: float, pack_rows: bool, entropy_error: bool,
                        chunk_rows: int = 1 << 20) -> dict:
        """One epoch whose samples arrive from (pinned) host memory: row chunks are copied on a side
        stream while the previous chunk's fp16 shadow and BMU search run, so only the update pass waits
        for the whole upload.  `host_X` is a float32 torch tensor [N, ldx] with the layout of the resident X."""
        torch = self.torch
        with torch.cuda.device(self.dev):
            S = self.samples
            X = S.X
            if tuple(host_X.shape) != tuple(X.shape) or host_X.dtype != torch.float32:
                raise ValueError("host_X must match the resident sample matrix (float32, same shape)")
            m, cur = self.M, self.W[self.cur]
            be = self._pick_backend(self.N, m)
            tensor = be[0] == nat.BMU_TENSOR
            need_lo = be[1] == 3
            S.row_perm = None  # the shadows are rebuilt chunk by chunk in natural sample order
            if tensor:
                S.reserve_shadows(need_lo)
            main = torch.cuda.current_stream(self.dev)
            if self._copy_stream is None:
                self._copy_stream = torch.cuda.Stream(self.dev)
            self._copy_stream.wait_stream(main)  # earlier readers of X are done before it is overwritten
            mpad = self._prepare_search(cur, m, be, 1)
            idx = self.idx.view(-1)[: self.N]
            for c0 in range(0, self.N, chunk_rows):
                c1 = min(self.N, c0 + chunk_rows)
                with torch.cuda.stream(self._copy_stream):
                    X[c0:c1].copy_(host_X[c0:c1], non_blocking=True)
                    ready = torch.cuda.Event()
                    ready.record(self._copy_stream)
                main.wait_event(ready)
                x16 = None
                if tensor:
                    x16 = (S.X16_hi[c0:c1], S.X16_lo[c0:c1] if need_lo else None, S.xnorm16[c0:c1])
                    self._prepare_x16(X[c0:c1], c1 - c0, *x16)
                self._bmu_search(X[c0:c1], c1 - c0, self.ldx, x16, cur, m, mpad, 1, False, idx[c0:c1], None, be,
                                 ws_key="bmu_chunk")
            part, hist = self._epoch_sums(entropy_error)
            self._accumulate(0, 0, self.N, X, idx, part, hist)
            return self._reduce_and_smooth(be, part, hist is not None, sigma, pack_rows, entropy_error)

    def epoch(self, sigma: float, pack_rows: bool, entropy_error: bool, _force_simt: bool = False) -> dict:
        """One training epoch: per chunk of the samples, fp16 shadows, BMU search and K2; then the all-reduce, K3 and
        the read-back.  Returns per-neuron error, counts, change."""
        torch = self.torch
        with torch.cuda.device(self.dev):
            S, m, cur = self.samples, self.M, self.W[self.cur]
            # the backend follows the whole sample count: small chunks must not turn the tensor search into the SIMT one
            be = (nat.BMU_SIMT, 0) if _force_simt else self._pick_backend(self.N, m)
            eligible = [self._select_eligible(c1 - c0, m, be) for c0, c1 in S.chunks]
            # the selective search needs the samples in sorted order, i.e. the winners of an earlier epoch
            selective = [e and S.has_order(c) for c, e in enumerate(eligible)]
            mpad = self._prepare_search(cur, m, be, 1, map_order=any(selective))
            part, hist = self._epoch_sums(entropy_error)
            idx = self.idx.view(-1)[: self.N]

            def body(c, c0, c1, x):
                x16, perm = S.shadows(c, x, be, selective[c])
                self._bmu_search(x, c1 - c0, self.ldx, x16, cur, m, mpad, 1, False, idx[c0:c1], None, be,
                                 row_perm=perm, selective=selective[c])
                S.after_k2(c, self._accumulate(c, c0, c1, x, idx, part, hist), eligible[c])

            S.chunk_pass(body)
            return self._reduce_and_smooth(be, part, hist is not None, sigma, pack_rows, entropy_error)

    def _epoch_sums(self, entropy_error: bool):
        """The epoch's K2 sums `part` and class histogram (None unless the entropy error needs it)."""
        m = self.M
        use_hist = entropy_error and self.labels is not None
        return self.part[: m * self.ldx + 3 * m], self.class_hist[:m] if use_hist else None

    def _accumulate(self, c: int, c0: int, c1: int, x, idx, part, hist):
        """K2 over chunk c (rows x of samples c0..c1, winners idx[c0:c1]).  Chunk 0 writes the epoch's `part` and class
        histogram `hist` (None: no histogram), later chunks write the chunk buffers, which are then added.  Returns
        the chunk's samples grouped by winner (chunk-local int32 [c1 - c0])."""
        n, m, first = c1 - c0, self.M, c == 0
        k_part = part if first else self._cpart[: part.numel()]
        k_hist = hist if first or hist is None else self._chist[:m]
        labels = self.labels[c0:c1] if hist is not None else None
        weight = self.weight[c0:c1] if self.weight is not None else None
        acc = nat.AccumulateArgs()
        acc.d_X, acc.N, acc.D, acc.ldx = x.data_ptr(), n, self.ldx, self.ldx
        acc.d_bmu, acc.d_W, acc.M = idx[c0:c1].data_ptr(), self.W[self.cur].data_ptr(), m
        acc.inv_total_variance = 1.0 / self.total_variance if self.total_variance > 0 else float("inf")
        acc.d_part = k_part.data_ptr()
        acc.d_labels = labels.data_ptr() if labels is not None else None
        acc.n_classes = self.n_classes if labels is not None else 0
        acc.d_class_hist = k_hist.data_ptr() if labels is not None and weight is None else None
        ws = self._workspace("acc", self.lib.dbgsom_accumulate_workspace_bytes(n, m, self.ldx))
        acc.d_workspace, acc.workspace_bytes = ws.data_ptr(), ws.numel()
        with self._Phase(self, "accumulate"):
            if weight is None:
                nat.check(self.lib.dbgsom_accumulate(acc, self._stream()), "dbgsom_accumulate")
            else:
                nat.check(
                    self.lib.dbgsom_accumulate_weighted(
                        acc, weight.data_ptr(), k_hist.data_ptr() if labels is not None else None, self._stream()
                    ),
                    "dbgsom_accumulate_weighted",
                )
        self.launches += (10 if m <= 24576 else 8) + (1 if labels is not None else 0)  # stable scatter: 3 kernels
        if not first:
            with self._Phase(self, "chunk_sum"):
                part.add_(k_part)
                if hist is not None:
                    hist.add_(k_hist)
        off = int(self.lib.dbgsom_accumulate_perm_offset(n, m))
        return ws[off : off + 4 * n].view(self.torch.int32)

    def _reduce_and_smooth(self, be, part, use_hist: bool, sigma: float, pack_rows: bool, entropy_error: bool) -> dict:
        """All-reduce of the epoch sums -> K3 -> read-back."""
        torch = self.torch
        m, cur = self.M, self.W[self.cur]
        # the one collective of the path: per-neuron partial sums (+ class histogram)
        with self._Phase(self, "allreduce"):
            self.comm.allreduce_(part)
            if use_hist:
                self.comm.allreduce_(self.class_hist[:m])

        # K3
        lut = np.exp(-(np.arange(self.hop_max + 1, dtype=np.float64) ** 2 / (2 * sigma**2)))
        d_lut = torch.from_numpy(lut).to(self.dev)
        out = self.W[self.cur ^ 1]
        sm = nat.SmoothArgs()
        sm.d_part, sm.d_hop, sm.ldh = part.data_ptr(), self.hop.data_ptr(), self.ldh
        sm.d_kernel_lut, sm.lut_len = d_lut.data_ptr(), int(lut.size)
        sm.M, sm.D, sm.pack_rows = m, self.ldx, int(bool(pack_rows))
        sm.d_W_in, sm.d_W_out, sm.d_change = cur.data_ptr(), out.data_ptr(), self.change.data_ptr()
        ws2 = self._workspace("smooth", self.lib.dbgsom_smooth_workspace_bytes(m, self.ldx))
        sm.d_workspace, sm.workspace_bytes = ws2.data_ptr(), ws2.numel()
        # Large maps on several GPUs: every rank smooths its own row range and the rows are all-gathered
        # (M^2 D flops / world instead of redundantly; the gathered copies are bit-identical on all ranks).
        world = self.comm.world if self.comm.enabled else 1
        rows_per = -(-m // world)
        shard_rows = world > 1 and m * m * self.ldx >= self.K3_SHARD_MIN_WORK and rows_per * world <= out.shape[0]
        if shard_rows:
            sm.row_begin = min(self.comm.rank * rows_per, m)
            sm.row_end = min(sm.row_begin + rows_per, m)
        with self._Phase(self, "smooth"):
            if not shard_rows or sm.row_end > sm.row_begin:
                nat.check(self.lib.dbgsom_smooth(sm, self._stream()), "dbgsom_smooth")
            else:
                self.change.zero_()
        self.launches += 7
        if shard_rows:
            with self._Phase(self, "allgather"):
                flat = out[: rows_per * world]
                mine = flat[self.comm.rank * rows_per : (self.comm.rank + 1) * rows_per]
                self.comm.dist.all_gather_into_tensor(flat, mine)
                self.comm.allreduce_(self.change)
        self.cur ^= 1
        self.n_previous_rows = m

        # one small D2H (syncs): [sk | n | E | change | wmax]
        tail = torch.cat([part[m * self.ldx :], self.change, self.wmax.double()]).cpu().numpy()
        counts, err, change = tail[m : 2 * m], tail[2 * m : 3 * m], float(tail[3 * m])
        if be[0] == nat.BMU_TENSOR and not tail[3 * m + 4] < 65000.0:
            # a prototype left the fp16 range of the shadow (far outside the data hull): its
            # scores were clamped, so redo this epoch on the fp32 path from the same state
            self.cur ^= 1
            self.fp32_reruns += 1
            return self.epoch(sigma, pack_rows, entropy_error, _force_simt=True)
        if use_hist:
            err = class_entropy(self.class_hist[:m].cpu().numpy())
        self.last_bmu_stats = None
        return {"error": err, "counts": counts, "change": change}

    def last_winners_host(self) -> np.ndarray:
        """BMU index of every local sample in the last `epoch` (int64 [N]; tests, diagnostics)."""
        return self.idx.view(-1)[: self.N].cpu().numpy().astype(np.int64)

    def bmu_stats_host(self, reset: bool = True) -> dict:
        """Cumulative re-score statistics of all BMU searches since the last reset."""
        s = self.bmu_stats.cpu().numpy()
        if reset:
            self.bmu_stats.zero_()
        out = {"ambiguous": int(s[0]), "flagged": int(s[1]), "candidates": int(s[2]), "full_rescans": int(s[3]),
               "refined_tiles": int(s[4]), "row_tile_pairs": int(s[5]), "fp32_reruns": int(self.fp32_reruns),
               "selective_searches": self._epoch_kinds["selective"], "classic_searches": self._epoch_kinds["classic"]}
        # MMA work of the top-1 three-pass searches in units of one fp16 pass over all (sample, prototype) pairs:
        # classic = 3; selective = 1 (FLAG pass) + 3 x the share of (row-tile pair, column tile) products refined
        n_sel, n_cls = out["selective_searches"], out["classic_searches"]
        if n_sel + n_cls:
            share = 0.0
            if s[5] > 0 and self.M > 0:
                share = float(s[4]) * self.select_granule / (float(s[5]) * _round_up(self.M, 256))
            out["refined_share"] = share
            out["mma_passes"] = (n_sel * (1.0 + 3.0 * share) + 3.0 * n_cls) / (n_sel + n_cls)
        if reset:
            self.fp32_reruns = 0
            self._epoch_kinds = {"selective": 0, "classic": 0}
        return out

    def bmu_train(self, n_bmu: int, previous: bool = False):
        """BMUs of the training samples against the current (or pre-update) prototypes."""
        with self.torch.cuda.device(self.dev):
            W = self.W[self.cur ^ 1] if previous else self.W[self.cur]
            m = self.n_previous_rows if previous else self.M
            n_bmu = min(n_bmu, m)
            dist_h = np.empty((self.N, n_bmu), dtype=np.float64)
            idx_h = np.empty((self.N, n_bmu), dtype=np.int64)

            def out(c, c0, c1, idx, dist):
                dist_h[c0:c1], idx_h[c0:c1] = dist.cpu().numpy(), idx.cpu().numpy()

            self._bmu_pass(W, m, n_bmu, self.strict_ties, out)
            return dist_h, idx_h

    def _bmu_pass(self, W, m: int, n_bmu: int, strict: bool, out) -> None:
        """BMU search of the training samples against W: per chunk, the chunk's winners idx int32 [n, n_bmu] and
        distances dist float64 [n, n_bmu] go to out(c, c0, c1, idx, dist), which enqueues what reads them before the
        next chunk overwrites them.  With one chunk they are the whole [N, n_bmu] results."""
        torch = self.torch
        be = self._pick_backend(self.N, m)
        mpad = self._prepare_search(W, m, be, n_bmu)
        rows = max((c1 - c0 for c0, c1 in self.samples.chunks), default=0)
        idx_buf = torch.empty((rows, n_bmu), dtype=torch.int32, device=self.dev)
        dist_buf = torch.empty((rows, n_bmu), dtype=torch.float64, device=self.dev)

        def body(c, c0, c1, x):
            n = c1 - c0
            x16, perm = self.samples.shadows(c, x, be, None)
            idx, dist = idx_buf[:n], dist_buf[:n]
            self._bmu_search(x, n, self.ldx, x16, W, m, mpad, n_bmu, True, idx, dist, be, strict=strict, row_perm=perm)
            out(c, c0, c1, idx, dist)

        self.samples.chunk_pass(body)

    # ------------------------------------------------------------------ post-training passes
    def final_statistics(self, positions: np.ndarray, degrees: np.ndarray) -> dict:
        """Everything `fit` measures after the loop, reduced on the device (and over ranks):
        one top-2 BMU search on the PRE-update prototypes (dbgsom/BaseSom.py:116-119 see the
        stale `weights_`) feeds the topographic error (:924-953), the quantisation error (:904-922)
        and the node statistics (:181-211); the u-matrix (:320-337) uses the updated prototypes."""
        torch = self.torch
        with torch.cuda.device(self.dev):
            m = self.n_previous_rows  # the samples are searched below, once the bandwidth is known
            n_bmu = min(2, m)
            M, cur = self.M, self.W[self.cur]
            total = float(np.sum(degrees))
            if total > 0:
                colw = torch.from_numpy(np.ascontiguousarray(degrees, dtype=np.float64) / total).to(self.dev)
                avg = torch.empty(M, dtype=torch.float64, device=self.dev)
                nat.check(
                    self.lib.dbgsom_umatrix(cur.data_ptr(), M, self.ldx, self.ldx, colw.data_ptr(), avg.data_ptr(), self._stream()),
                    "dbgsom_umatrix",
                )
                self.launches += 2
                avg_host = avg.cpu().numpy()
            else:
                avg_host = np.full(M, np.nan)
            bandwidth = float(avg_host.mean())
            pos = torch.from_numpy(np.ascontiguousarray(positions[:m], dtype=np.int32)).to(self.dev)
            out = torch.empty(2 + 2 * m, dtype=torch.float64, device=self.dev)
            ok = bandwidth > 0 and math.isfinite(bandwidth)

            def stats(c, c0, c1, idx, dist):
                # chunk 0 writes `out`, later chunks a chunk buffer that is added into it
                k_out = out if c == 0 else torch.empty_like(out)
                w = self.weight[c0:c1] if self.weight is not None else None
                self._node_stats(idx, dist, n_bmu, c1 - c0, pos, m, bandwidth if ok else 1.0, w, k_out)
                if c:
                    out.add_(k_out)

            self._bmu_pass(self.W[self.cur ^ 1], m, n_bmu, True, stats)
            self.comm.allreduce_(out)
            o = out.cpu().numpy()
            dens = o[2 + m :].copy()
            if not ok:
                dens[:] = np.nan
            return {"te_count": float(o[0]), "qe_sum": float(o[1]), "hits": o[2 : 2 + m].copy(), "dens_sum": dens,
                    "avg_dist": avg_host, "weights": self.weights(), "n_rows": m}

    def _node_stats(self, idx, dist, n_bmu: int, n: int, pos, m: int, bandwidth: float, weight, out) -> None:
        if weight is None:
            nat.check(
                self.lib.dbgsom_node_stats(
                    idx.data_ptr(), n_bmu, dist.data_ptr(), n_bmu, n, pos.data_ptr(), m,
                    bandwidth, out.data_ptr(), self._stream(),
                ),
                "dbgsom_node_stats",
            )
        else:
            nat.check(
                self.lib.dbgsom_node_stats_weighted(
                    idx.data_ptr(), n_bmu, dist.data_ptr(), n_bmu, n, pos.data_ptr(), m,
                    bandwidth, weight.data_ptr(), out.data_ptr(), self._stream(),
                ),
                "dbgsom_node_stats_weighted",
            )
        self.launches += 2

    def final_winners(self) -> None:
        """Top-1 BMU of the training samples on the current (reduced) map; stays on the device."""
        with self.torch.cuda.device(self.dev):
            # one chunk: the pass's own [N, 1] winners are kept
            chunked = len(self.samples.chunks) > 1
            self._final_idx = self.torch.empty((self.N, 1), dtype=self.torch.int32, device=self.dev) if chunked else None

            def keep(c, c0, c1, idx, dist):
                if chunked:
                    self._final_idx[c0:c1].copy_(idx)
                else:
                    self._final_idx = idx

            self._bmu_pass(self.W[self.cur], self.M, 1, True, keep)

    def winners_host(self) -> np.ndarray:
        return self._final_idx[:, 0].cpu().numpy().astype(np.int64)

    def label_histogram(self, n_classes: int):
        """Class counts [M, C] and first global sample index [M, C] of every (winner, class) cell of the
        last `final_winners` search, reduced over ranks (dbgsom/SomClassifier.py:130-152).  Weighted fits: the
        counts are weight sums and `first` ignores zero-weight samples.  Per chunk of the samples: counts added in
        chunk order, `first` the minimum over the chunks."""
        torch = self.torch
        with torch.cuda.device(self.dev):
            m, weighted = self.M, self.weight is not None
            for c, (c0, c1) in enumerate(self.samples.chunks):
                n, idx = c1 - c0, self._final_idx[c0:c1]
                counts = torch.empty((m, n_classes), dtype=torch.float64 if weighted else torch.int32, device=self.dev)
                k_first = torch.empty((m, n_classes), dtype=torch.int64, device=self.dev)
                if weighted:
                    ws = self._workspace("labels", self.lib.dbgsom_label_hist_weighted_workspace_bytes(n, m))
                    nat.check(
                        self.lib.dbgsom_label_hist_weighted(
                            idx.data_ptr(), self.labels[c0:c1].data_ptr(), self.weight[c0:c1].data_ptr(), n,
                            self.sample_offset + c0, m, n_classes, counts.data_ptr(), k_first.data_ptr(),
                            ws.data_ptr(), ws.numel(), self._stream(),
                        ),
                        "dbgsom_label_hist_weighted",
                    )
                else:
                    nat.check(
                        self.lib.dbgsom_label_hist(
                            idx.data_ptr(), int(idx.shape[1]), self.labels[c0:c1].data_ptr(), n, self.sample_offset + c0,
                            m, n_classes, counts.data_ptr(), k_first.data_ptr(), self._stream(),
                        ),
                        "dbgsom_label_hist",
                    )
                self.launches += 3
                if c == 0:  # int32 counts are summed as int64
                    total, first = counts.to(torch.float64 if weighted else torch.int64), k_first
                else:
                    total.add_(counts)
                    torch.minimum(first, k_first, out=first)
            self.comm.allreduce_(total)
            self.comm.allreduce_(first, "min")
            return total.cpu().numpy().astype(np.float64), first.cpu().numpy()

    def bmu(self, X: np.ndarray, W: np.ndarray, n_bmu: int):
        """Stand-alone BMU search (predict path): host samples against host prototypes.

        Samples whose upload would not fit in device memory (or `stream_rows` > 0) are searched in row chunks; the
        shadow shift and scale still come from all of X, so every row gets the winner and distance of one call."""
        torch = self.torch
        with torch.cuda.device(self.dev):
            n, d = int(X.shape[0]), int(X.shape[1])
            if d != W.shape[1]:
                raise ValueError(f"X has {d} features, the map has {W.shape[1]}")
            rows = self._plan_rows(n, d, 0, False, capacity=W.shape[0])
            chunks = [(0, n)] if rows is None else streaming.chunk_bounds(n, rows)
            self.N, self.D = chunks[0][1] - chunks[0][0], d
            self.ldx = _round_up(d, 4)
            self.ld16 = _round_up(self.ldx, 64)
            self.labels, self.n_classes = None, 0
            self.W = None
            self._alloc_map(W.shape[0])
            self.cur = 0
            self.set_map(np.asarray(W))
            # shadows for the tensor path: centre on the prototypes' mean, scale from both operands
            be = self._pick_backend(n, self.M)
            tensor = be[0] == nat.BMU_TENSOR
            if tensor:
                centre = np.asarray(W, dtype=np.float64).mean(axis=0)
                shift = np.zeros(self.ldx, dtype=np.float32)
                shift[:d] = centre
                self.shift = torch.from_numpy(shift).to(self.dev)
                x_max = max(float(np.abs(np.asarray(X[c0:c1]) - centre).max()) for c0, c1 in chunks)
                maxabs = float(max(x_max, np.abs(np.asarray(W) - centre).max()))
                self.scale = 1.0 if not (maxabs > 0 and math.isfinite(maxabs)) else 2.0 ** math.floor(
                    math.log2(2.0**14 / maxabs)
                )  # both operands are in hand here, so the bound is exact
            else:
                self.shift = torch.zeros(self.ldx, dtype=torch.float32, device=self.dev)
                self.scale = 1.0
            n_bmu = min(n_bmu, self.M)
            dist_h = np.empty((n, n_bmu), dtype=np.float64)
            idx_h = np.empty((n, n_bmu), dtype=np.int64)
            for c0, c1 in chunks:
                self.N = c1 - c0
                x = self._upload_matrix(np.asarray(X[c0:c1]))
                x16, _ = ResidentSamples(self, x).shadows(0, x, be, None)
                idx = torch.empty((self.N, n_bmu), dtype=torch.int32, device=self.dev)
                dist = torch.empty((self.N, n_bmu), dtype=torch.float64, device=self.dev)
                self._run_bmu(x, self.N, self.ldx, x16, self.W[0], self.M, n_bmu, True, idx, dist, backend=be)
                dist_h[c0:c1], idx_h[c0:c1] = dist.cpu().numpy(), idx.cpu().numpy()
            return dist_h, idx_h

    # ------------------------------------------------------------------ sparse coding (transform)
    def sparse_code(self, Xn: np.ndarray, Wn: np.ndarray, max_iter: int = 1000) -> np.ndarray:
        """Non-negative LARS-lasso code of the row-normalised samples `Xn` [N, D] over the row-normalised
        prototypes `Wn` [M, D] (what `SparseCoder(..., "lasso_lars", positive_code=True, transform_alpha=0)`
        computes in dbgsom/BaseSom.py:241-268).  Gram matrix and correlations are two float64 GEMMs (cuBLAS
        through torch), the per-sample paths run in `dbgsom_sparse_code`, one CUDA thread per sample."""
        torch = self.torch
        n, d = int(Xn.shape[0]), int(Xn.shape[1])
        m = int(Wn.shape[0])
        if Wn.shape[1] != d:
            raise ValueError(f"X has {d} features, the map has {Wn.shape[1]}")
        out = np.empty((n, m), dtype=np.float64)
        with torch.cuda.device(self.dev):
            W = torch.from_numpy(np.ascontiguousarray(Wn, dtype=np.float64)).to(self.dev)
            gram = (W @ W.T).contiguous()
            chunk = max(1024, min(n, int((1 << 30) // (8 * m))))  # cov + code of a chunk: 2 GiB at most
            budget = 2 << 30  # scratch of the per-thread paths
            for c0 in range(0, n, chunk):
                c1 = min(n, c0 + chunk)
                nc = c1 - c0
                X = torch.from_numpy(np.ascontiguousarray(Xn[c0:c1])).to(self.dev).to(torch.float64)
                cov = (X @ W.T).contiguous()
                code = torch.zeros((nc, m), dtype=torch.float64, device=self.dev)
                status = torch.zeros(nc, dtype=torch.int32, device=self.dev)
                rows, n_rows = None, nc
                for cap in (min(m, 32), min(m, 128), min(m, 1024)):
                    per_thread = self.lib.dbgsom_sparse_code_workspace_bytes(1, m, cap)
                    threads = max(128, min(-(-n_rows // 128) * 128, (budget // per_thread) // 128 * 128))
                    ws = self._workspace("lars", self.lib.dbgsom_sparse_code_workspace_bytes(threads, m, cap))
                    nat.check(
                        self.lib.dbgsom_sparse_code(
                            gram.data_ptr(), cov.data_ptr(), n_rows, m, d, int(max_iter), cap,
                            rows.data_ptr() if rows is not None else None, code.data_ptr(), status.data_ptr(),
                            ws.data_ptr(), ws.numel(), self._stream(),
                        ),
                        "dbgsom_sparse_code",
                    )
                    self.launches += 1
                    rows = torch.nonzero(status & 1).to(torch.int32).view(-1).contiguous()
                    n_rows = int(rows.numel())
                    if n_rows == 0 or cap == m:
                        break
                if n_rows:
                    raise nat.NativeError(f"{n_rows} samples need more than 1024 active atoms in the LARS path")
                out[c0:c1] = code.cpu().numpy()
        return out

    # ------------------------------------------------------------------ host-side reductions
    def allreduce_scalars(self, vals):
        if not (self.comm.enabled and self.comm.world > 1):
            return list(vals)
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        return self.comm.allreduce_(t).cpu().tolist()

    def allreduce_arrays(self, arrs, op: str = "sum"):
        if not (self.comm.enabled and self.comm.world > 1):
            return list(arrs)
        out = []
        for a in arrs:
            t = self.torch.from_numpy(np.ascontiguousarray(a)).to(self.dev)
            out.append(self.comm.allreduce_(t, op).cpu().numpy())
        return out
