"""The device against tests/reference_semantics.py: the getter casts of fixed_batch_kernel (K1-K4) and the VARCHAR
renderings of render_text_kernel (K7) on the edge sets of tests/test_reference_cpu.py.

Every edge value is placed at row 0 of a chunk, inside the 16-byte vectors, in the scalar tail of a chunk (the last
`count % R` rows) and, for the narrow conversions, in chunks converted together by the grouped path; on full and
ragged chunk patterns, with NULLs that have garbage under them.  The bulk sweeps (float32 bit patterns, random day
numbers and microseconds) compare the device with the oracle, which test_reference_cpu.py pins on the same kinds of
values."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import oracle  # noqa: E402
import reference_semantics as rs  # noqa: E402
from duckdb_mbt_b200 import chunks as ch  # noqa: E402
from test_reference_cpu import (EDGE_COLUMNS, TEXT_COLUMNS, TS_MIN_US, edge_batch, expected_texts,  # noqa: E402
                                position_counts, value_mismatches)


def _device_mod():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from duckdb_mbt_b200 import device
    return device


@pytest.fixture(scope="module")
def ctx():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from duckdb_mbt_b200 import arrow_result as ar
    c = ar.GpuContext(0)
    yield c
    c.close()


def _result(ctx, batch):
    from duckdb_mbt_b200 import arrow_result as ar
    return ar.ArrowResult.from_chunks(ctx, batch)


def _check_casts(dev, cols, counts, rng=None, null_every=0):
    """every getter cast of every edge column in one plan (one launch per distinct conversion)"""
    batch, idxs, valid = edge_batch(cols, counts, rng, null_every)
    specs = [(j, dst) for j, col in enumerate(cols) for dst in col[5]]
    db = dev.DeviceBatch(batch)
    plan = db.plan_fixed(specs, bitmap=True, valid_bytes=False)
    db.run_fixed(plan)
    torch.cuda.synchronize()
    for o in plan[0]:
        dst = o.op & 0xFF
        rows, bad = value_mismatches(cols[o.col], dst, dev.to_numpy(o.values), idxs[o.col], valid)
        if rows.size:
            pytest.fail(f"{cols[o.col][0]} dst={dst}: device differs from the reference for {bad[:8]} (first row {rows[0]})")


@pytest.mark.parametrize("n,pattern", [(1, "full"), (2047, "full"), (2049, "full"), (2047, "ragged"), (50_000, "full"),
                                       (50_000, "ragged")])
def test_device_casts_match_the_references(n, pattern):
    dev = _device_mod()
    rng = np.random.default_rng(170 + n)
    counts = ch.chunk_counts(n, pattern, rng)
    _check_casts(dev, EDGE_COLUMNS, counts, rng, null_every=7 if n > 1 else 0)


def test_device_casts_at_every_position():
    """2E chunks of 2033 / 2047 rows per edge column: each edge value at a chunk's row 0, in the vector body and in
    the scalar tail of a chunk, for every rows-per-vector the column's conversions use"""
    dev = _device_mod()
    for col in EDGE_COLUMNS:
        _check_casts(dev, [col], position_counts(len(col[4])))


def _text_of(t, n):
    return [t.data[int(t.offsets[i]):int(t.offsets[i + 1])] for i in range(n)]


def _check_text(ctx, cols, counts, rng=None, null_every=0, per_cell=False):
    from duckdb_mbt_b200 import typed_result as tr
    batch, idxs, valid = edge_batch(cols, counts, rng, null_every)
    n = batch.nrows
    ora = oracle.OracleResult(batch)
    with _result(ctx, batch) as res:
        for j, col in enumerate(cols):
            exp = expected_texts(col, idxs[j])
            t = tr.text_column(res, j)
            got = _text_of(t, n)
            ok = np.ones(n, bool) if valid is None else valid
            assert np.array_equal(t.valid, ok), col[0]
            bad = [(col[4][idxs[j][i]], got[i], exp[i]) for i in range(n) if ok[i] and exp[i] is not None and got[i] != exp[i]]
            assert not bad, f"{col[0]}: (value, device, reference) {bad[:6]}"
            assert all(got[i] == b"" for i in range(n) if not ok[i]), col[0]
            for nullable in (False, True):
                blob = res.raw_column("string", j, nullable)
                assert blob == ora.get_column("string", j, nullable), (col[0], nullable)
                if valid is None and all(x is not None for x in exp):
                    stream = b"".join(x + b"\0" for x in exp)
                    want = np.asarray([n, len(stream)], dtype="<i4").tobytes() + stream + (b"\x01" * n if nullable else b"")
                    assert blob == want, (col[0], nullable)
        if per_cell:
            from duckdb_mbt_b200.query_result import query_per_cell
            p = query_per_cell(res)
            for j, col in enumerate(cols):
                exp = expected_texts(col, idxs[j])
                for i in range(n):
                    if exp[i] is not None:
                        assert p.rows[i][j] == exp[i].decode(), (col[0], col[4][idxs[j][i]])


def test_device_text_of_every_edge_value(ctx):
    """text_column, both string getters and the per-cell value symbol against the references, one row per edge value"""
    for col in TEXT_COLUMNS:
        _check_text(ctx, [col], ch.chunk_counts(len(col[4])), per_cell=True)


@pytest.mark.parametrize("n,pattern", [(2047, "full"), (2049, "full"), (50_000, "ragged")])
def test_device_text_with_nulls_and_ragged_chunks(ctx, n, pattern):
    rng = np.random.default_rng(270 + n)
    counts = ch.chunk_counts(n, pattern, rng)
    _check_text(ctx, TEXT_COLUMNS, counts, rng, null_every=7)


def test_device_float_text_sweep(ctx):
    """every 2^8-th float32 bit pattern, every float within 2^15 patterns of 1e-5, 1, 2^24 and 1e16 (both signs; both
    layouts at the 1e-5 / 1e16 boundaries) and every 61st subnormal: device text == oracle text.  The oracle renders
    a float in about 6 us, so it runs on slices of the sweep in threads (ctypes releases the GIL)."""
    from concurrent.futures import ThreadPoolExecutor
    pats = [np.arange(0, 2**32, 2**8, dtype=np.uint64).astype(np.uint32)]
    for v in (1e-5, 1.0, 2.0 ** 24, 1e16):
        run = np.arange(-2**15, 2**15, dtype=np.int64) + int(np.float32(v).view(np.uint32))
        pats += [run.astype(np.uint32), run.astype(np.uint32) | np.uint32(2**31)]
    pats.append(np.arange(1, 2**23, 61, dtype=np.uint32))
    vals = np.concatenate(pats).view(np.float32)
    vals = vals[~(np.isnan(vals) & np.signbit(vals))]
    n = vals.shape[0]

    def oracle_stream(part):
        c = ch.chunk_counts(part.shape[0])
        blob = oracle.OracleResult(ch.ChunkBatch(c, [ch.fixed_column("f", ch.T_FLOAT, part, c)])).get_column("string", 0)
        return blob[8:]

    oracle.lib()  # built and loaded before the threads
    parts = np.array_split(vals, 64)
    with ThreadPoolExecutor(max_workers=16) as pool:
        stream = b"".join(pool.map(oracle_stream, parts))
    counts = ch.chunk_counts(n)
    with _result(ctx, ch.ChunkBatch(counts, [ch.fixed_column("f", ch.T_FLOAT, vals, counts)])) as res:
        got = res.raw_column("string", 0, False)
    assert got[:8] == np.asarray([n, len(stream)], dtype="<i4").tobytes()
    if got[8:] != stream:
        cut = next(i for i in range(len(stream)) if got[8 + i] != stream[i])
        row = stream[:cut].count(b"\0")
        pytest.fail(f"float {float(vals[row])!r}: device {got[8:].split(bytes(1))[row]!r}, oracle {stream.split(bytes(1))[row]!r}")


def test_device_date_and_timestamp_sweep(ctx):
    """10^5 random int32 day numbers and int64 microseconds (DuckDB's whole finite range and the sentinels)"""
    rng = np.random.default_rng(8)
    n = 100_000
    days = rng.integers(-(2**31) + 2, 2**31 - 1, n, dtype=np.int64)
    days[: n // 2] = rng.integers(-800_000, 3_000_000, n // 2)
    days[[7, 77, 777]] = [2**31 - 1, -(2**31 - 1), 0]
    micros = rng.integers(TS_MIN_US, 2**63 - 1, n, dtype=np.int64)
    micros[: n // 2] = rng.integers(-(10**17), 10**17, n // 2)
    micros[[7, 77]] = [2**63 - 1, -(2**63 - 1)]
    counts = ch.chunk_counts(n, "ragged", rng)
    valid = rng.random(n) > 0.1
    batch = ch.ChunkBatch(counts, [ch.fixed_column("d", ch.T_DATE, days.astype(np.int32), counts, valid=valid, garbage_rng=rng),
                                   ch.fixed_column("t", ch.T_TIMESTAMP, micros, counts, valid=valid, garbage_rng=rng),
                                   ch.fixed_column("z", ch.T_TIMESTAMP_TZ, micros, counts, valid=valid, garbage_rng=rng)])
    ora = oracle.OracleResult(batch)
    from duckdb_mbt_b200 import typed_result as tr
    with _result(ctx, batch) as res:
        for j in range(3):
            for nullable in (False, True):
                assert res.raw_column("string", j, nullable) == ora.get_column("string", j, nullable), (j, nullable)
        d, t = _text_of(tr.text_column(res, 0), n), _text_of(tr.text_column(res, 1), n)
    for i in list(rng.integers(0, n, 2000)) + [7, 77]:
        if valid[i]:
            assert d[i].decode() == rs.render_date(int(days[i])), int(days[i])
            assert t[i].decode() == rs.render_timestamp(int(micros[i])), int(micros[i])
