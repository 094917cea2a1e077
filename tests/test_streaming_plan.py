"""Chunk planning of streamed fits (dbgsom_b200/streaming.py): pure host arithmetic, no device."""

import numpy as np
import pytest

from dbgsom_b200 import streaming as S


def acc_ws(n, m, d):  # shapes like the library's: per-sample buckets + per-neuron tables
    return 12 * n + 64 * m + 8 * d


def bmu_ws(n, n_bmu):
    return 40 * n * n_bmu + 4096


ARGS = dict(capacity=264, n_classes=10, weighted=True, acc_ws_bytes=acc_ws, bmu_ws_bytes=bmu_ws)


@pytest.mark.parametrize("n,d", [(1000, 64), (100_000, 256), (2_000_000, 4096)])
def test_resident_exactly_when_the_resident_footprint_fits(n, d):
    need = S.resident_bytes(n, d, **ARGS)
    assert S.plan_stream(n, d, free_bytes=need, **ARGS) is None
    rows = S.plan_stream(n, d, free_bytes=need - 1, **ARGS)
    assert rows is not None and rows > 0


@pytest.mark.parametrize("n,d,free", [(1_000_000, 128, 200 << 20), (300_000, 4096, 3 << 30), (50_000, 7, 10 << 20)])
def test_chunks_are_multiples_of_256_that_fit(n, d, free):
    rows = S.plan_stream(n, d, free_bytes=free, **ARGS)
    assert rows is not None and rows % S.ROW_GRANULE == 0
    assert S.streamed_bytes(rows, n, d, **ARGS) <= free
    ldx = -(-d // 4) * 4
    # the largest that fits (up to the chunk-size cap)
    cap_rows = min(-(-n // 256) * 256, S.MAX_CHUNK_BYTES // (4 * ldx) // 256 * 256)
    assert rows == cap_rows or S.streamed_bytes(rows + S.ROW_GRANULE, n, d, **ARGS) > free
    chunks = S.chunk_bounds(n, rows)
    assert chunks[0][0] == 0 and chunks[-1][1] == n
    assert all(b - a == rows for a, b in chunks[:-1]) and 0 < chunks[-1][1] - chunks[-1][0] <= rows
    assert all(chunks[i][1] == chunks[i + 1][0] for i in range(len(chunks) - 1))


def test_last_chunk_is_ragged():
    chunks = S.chunk_bounds(200_000, 76_800)
    assert [b - a for a, b in chunks] == [76_800, 76_800, 46_400]


def test_streaming_beats_resident_memory_per_sample():
    n, d = 10_000_000, 256
    res = S.resident_bytes(n, d, **ARGS)
    st = S.streamed_bytes(1 << 16, n, d, **ARGS)
    assert st < res / 20


def test_a_fit_that_cannot_stream_raises_memory_error():
    n, d = 10_000_000, 128
    floor = S.streamed_bytes(S.ROW_GRANULE, n, d, **ARGS)
    assert S.plan_stream(n, d, free_bytes=floor, **ARGS) == S.ROW_GRANULE
    with pytest.raises(MemoryError, match="bytes per sample"):
        S.plan_stream(n, d, free_bytes=floor - 1, **ARGS)
    with pytest.raises(MemoryError):
        S.plan_stream(n, d, free_bytes=0, **ARGS)


def test_map_capacity_counts_the_hop_matrix():
    small = S.resident_bytes(1000, 64, **{**ARGS, "capacity": 1000})
    big = S.resident_bytes(1000, 64, **{**ARGS, "capacity": 20000})
    assert big - small >= 2 * (20224**2 - 1024**2)


def test_env_switch_overrides_the_plan(monkeypatch):
    monkeypatch.setenv("DBGSOM_STREAM_ROWS", "1000")
    assert S.stream_rows_from_env() == 1024
    monkeypatch.setenv("DBGSOM_STREAM_ROWS", "512")
    assert S.stream_rows_from_env() == 512
    monkeypatch.setenv("DBGSOM_STREAM_ROWS", "0")
    assert S.stream_rows_from_env() == 0
    monkeypatch.delenv("DBGSOM_STREAM_ROWS")
    assert S.stream_rows_from_env() == 0


def test_engine_takes_the_switch_before_planning(monkeypatch):
    """DeviceEngine._plan_rows: a positive `stream_rows` wins over the free-memory plan (no device is touched)."""
    from dbgsom_b200.engine import DeviceEngine

    eng = DeviceEngine.__new__(DeviceEngine)
    eng.stream_rows = 700
    eng.capacity_hint = 64
    eng.free_device_bytes = lambda: pytest.fail("the plan must not run when streaming is forced")
    assert eng._plan_rows(10_000, 32, 0, False) == 768
    eng.stream_rows = 0
    eng.free_device_bytes = lambda: 1 << 40
    eng.lib = type("Lib", (), {"dbgsom_accumulate_workspace_bytes": staticmethod(acc_ws),
                               "dbgsom_bmu_workspace_bytes": staticmethod(bmu_ws)})()
    assert eng._plan_rows(10_000, 32, 0, False) is None
    eng.free_device_bytes = lambda: 16 << 20
    rows = eng._plan_rows(1_000_000, 32, 0, False)
    assert rows is not None and rows % 256 == 0


def test_estimator_passes_its_map_capacity_to_the_engine(monkeypatch):
    from dbgsom_b200 import SomVQ
    from dbgsom_b200 import engine as E

    seen = {}
    monkeypatch.setattr(E, "DeviceEngine", lambda **kw: seen.update(kw) or "engine")
    assert SomVQ(max_neurons=300)._make_engine() == "engine"
    assert seen["capacity_hint"] == SomVQ(max_neurons=300)._capacity_hint() == 664


def test_staging_converts_float64_like_the_resident_upload():
    """The host conversion the ring uses (numpy same_kind copy) rounds float64 to nearest float32, as torch's
    float64 -> float32 conversion of the resident upload does."""
    import torch

    rng = np.random.default_rng(0)
    X = rng.normal(size=(1000, 13)) * 10.0 ** rng.integers(-8, 8, size=(1000, 1))
    buf = np.zeros((1000, 16), dtype=np.float32)
    np.copyto(buf[:, :13], X, casting="same_kind")
    ref = torch.from_numpy(X).to(torch.float32).numpy()
    np.testing.assert_array_equal(buf[:, :13], ref)
    assert not buf[:, 13:].any()
