"""GPU parity, device API (L0): hand-written kernels vs the CPU oracle, bit-exact, on seeded
DuckDB-shaped chunk batches (full and ragged chunk patterns, NULL-pointer validity, garbage under
NULLs, inline/pointer strings)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import oracle  # noqa: E402
from duckdb_mbt_b200 import chunks as ch  # noqa: E402


def _device_mod():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from duckdb_mbt_b200 import device
    return device


def _check_fixed(dev_mod, batch, specs, valid_bytes=True):
    db = dev_mod.DeviceBatch(batch)
    plan = db.plan_fixed(specs, bitmap=True, valid_bytes=valid_bytes)
    db.run_fixed(plan)
    torch.cuda.synchronize()
    ora = oracle.OracleResult(batch)
    n = batch.nrows
    for o in plan[0]:
        dst = o.op & 0xFF if o.op != ch.OP_VALIDITY_ONLY else None
        if dst is None:
            _, bm, vb, nc = ora.arrow_fixed(o.col, ch.D_SAME, 16, want_values=False)
        else:
            ev, bm, vb, nc = ora.arrow_fixed(o.col, dst, o.width)
            got = dev_mod.to_numpy(o.values)[: ev.shape[0]]
            assert np.array_equal(got, ev), f"values differ col={o.col} op={o.op:#x}"
        got_bm = dev_mod.to_numpy(o.bitmap)[: bm.shape[0]]
        assert np.array_equal(got_bm, bm), f"bitmap differs col={o.col}"
        if valid_bytes:
            assert np.array_equal(dev_mod.to_numpy(o.valid_bytes)[:n], vb), f"validity bytes differ col={o.col}"
        assert int(dev_mod.to_numpy(o.null_count, np.uint64)[0]) == nc


def _mixed_batch(n, pattern, seed):
    rng = np.random.default_rng(seed)
    counts = ch.chunk_counts(n, pattern, rng)
    def valid(p=0.25):
        return rng.random(n) >= p
    cols = [
        ch.fixed_column("b", ch.T_BOOLEAN, rng.integers(0, 2, n).astype(np.uint8), counts, valid=valid(), garbage_rng=rng),
        ch.fixed_column("i8", ch.T_TINYINT, rng.integers(-128, 128, n).astype(np.int8), counts, valid=valid(), garbage_rng=rng),
        ch.fixed_column("i16", ch.T_SMALLINT, rng.integers(-2**15, 2**15, n).astype(np.int16), counts),
        ch.fixed_column("i32", ch.T_INTEGER, rng.integers(-2**31, 2**31, n).astype(np.int32), counts, valid=valid(), garbage_rng=rng),
        ch.fixed_column("i64", ch.T_BIGINT, rng.integers(-2**63, 2**63 - 1, n, dtype=np.int64), counts, valid=valid(), garbage_rng=rng),
        ch.fixed_column("u8", ch.T_UTINYINT, rng.integers(0, 256, n).astype(np.uint8), counts),
        ch.fixed_column("u16", ch.T_USMALLINT, rng.integers(0, 2**16, n).astype(np.uint16), counts, valid=valid(), garbage_rng=rng),
        ch.fixed_column("u32", ch.T_UINTEGER, rng.integers(0, 2**32, n).astype(np.uint32), counts),
        ch.fixed_column("u64", ch.T_UBIGINT, rng.integers(0, 2**64 - 1, n, dtype=np.uint64), counts, valid=valid(), garbage_rng=rng),
        ch.fixed_column("f32", ch.T_FLOAT, (rng.standard_normal(n) * 1e3).astype(np.float32), counts, valid=valid(), garbage_rng=None),
        ch.fixed_column("f64", ch.T_DOUBLE, rng.standard_normal(n) * 1e6, counts, valid=valid(), garbage_rng=None),
        ch.fixed_column("huge", ch.T_HUGEINT, rng.integers(0, 256, (n, 16), dtype=np.uint8), counts, valid=valid(), garbage_rng=rng),
        ch.fixed_column("dec4", ch.T_DECIMAL, rng.integers(-9999, 10000, n).astype(np.int16), counts, valid=valid(), dec_width=4, dec_scale=1, garbage_rng=rng),
        ch.fixed_column("dec9", ch.T_DECIMAL, rng.integers(-10**9 + 1, 10**9, n).astype(np.int32), counts, valid=valid(), dec_width=9, dec_scale=2, garbage_rng=rng),
        ch.fixed_column("dec18", ch.T_DECIMAL, rng.integers(-10**18 + 1, 10**18, n, dtype=np.int64), counts, valid=valid(), dec_width=18, dec_scale=3, garbage_rng=rng),
        ch.fixed_column("date", ch.T_DATE, rng.integers(-200000, 200000, n).astype(np.int32), counts, valid=valid(), garbage_rng=rng),
        ch.fixed_column("ts_s", ch.T_TIMESTAMP_S, rng.integers(-10**10, 10**10, n, dtype=np.int64), counts, valid=valid(), garbage_rng=rng),
        ch.fixed_column("ts_ms", ch.T_TIMESTAMP_MS, rng.integers(-10**13, 10**13, n, dtype=np.int64), counts),
        ch.fixed_column("ts_ns", ch.T_TIMESTAMP_NS, rng.integers(-10**18, 10**18, n, dtype=np.int64), counts, valid=valid(), garbage_rng=rng),
        ch.fixed_column("iv", ch.T_INTERVAL, rng.integers(0, 256, (n, 16), dtype=np.uint8), counts, valid=valid(), garbage_rng=rng),
        ch.fixed_column("uuid", ch.T_UUID, rng.integers(0, 256, (n, 16), dtype=np.uint8), counts),
    ]
    return ch.ChunkBatch(counts, cols)


ALL_SPECS = (
    [(c, ch.D_SAME) for c in range(21)]
    + [(c, ch.D_I64) for c in range(0, 12)] + [(c, ch.D_I32_TRUNC) for c in range(0, 12)]
    + [(c, ch.D_F64) for c in range(0, 11)] + [(c, ch.D_BOOL_BYTE) for c in range(0, 11)]
    + [(0, ch.D_BOOL_BITS)]
    + [(c, ch.D_I128) for c in (11, 12, 13, 14)]
    + [(11, ch.D_F64), (11, ch.D_BOOL_BYTE), (20, ch.D_I64), (20, ch.D_I32_TRUNC), (20, ch.D_F64), (20, ch.D_BOOL_BYTE)]  # HUGEINT / 128-bit unsigned
    + [(c, d) for c in (12, 13, 14) for d in (ch.D_DEC_I64, ch.D_DEC_I32_TRUNC, ch.D_DEC_F64, ch.D_DEC_BOOL_BYTE)]
    + [(c, ch.D_I32_SAT) for c in range(1, 9)]
    + [(16, ch.D_TS_US_FROM_S), (17, ch.D_TS_US_FROM_MS), (18, ch.D_TS_US_FROM_NS)]
    + [(19, ch.D_MONTH_DAY_NANO), (15, ch.D_DATE_REF), (4, ch.OP_VALIDITY_ONLY)]
)


@pytest.mark.parametrize("n,pattern", [(1, "full"), (63, "full"), (2048, "full"), (2049, "full"),
                                       (10_000, "full"), (10_000, "ragged"), (50_001, "ragged")])
def test_fixed_all_ops(n, pattern):
    dev = _device_mod()
    _check_fixed(dev, _mixed_batch(n, pattern, seed=100 + n), ALL_SPECS)


def test_fixed_config_c1():
    dev = _device_mod()
    for variant_b in (False, True):
        b = ch.config_c1(100_000, variant_b=variant_b)
        _check_fixed(dev, b, [(0, ch.D_SAME), (1, ch.D_SAME), (2, ch.D_SAME), (0, ch.D_I32_TRUNC), (1, ch.D_F64), (2, ch.D_I64)])


def test_fixed_config_c4_shape():
    dev = _device_mod()
    b = ch.config_c4(30_000, ncols=9, pattern="ragged")
    specs = []
    for j, col in enumerate(b.columns):
        specs.append((j, ch.D_I128 if col.type_id == ch.T_DECIMAL else ch.D_SAME))
    _check_fixed(dev, b, specs, valid_bytes=False)


def _check_string(dev_mod, batch, col=0, modes=(0, 1, 2)):
    db = dev_mod.DeviceBatch(batch)
    ora = oracle.OracleResult(batch)
    for mode in modes:
        so = db.plan_string(col, mode)
        db.run_string(so)
        assert db.string_error(so) == 0
        eo, ed = ora.arrow_string(col, mode)
        got_o = dev_mod.to_numpy(so.offsets, np.int64 if mode == 1 else np.int32)[: eo.shape[0]]
        assert np.array_equal(got_o, eo), f"offsets differ mode={mode}"
        total = int(dev_mod.to_numpy(so.total, np.uint64)[0])
        assert total == ed.shape[0]
        assert np.array_equal(dev_mod.to_numpy(so.data)[:total], ed), f"data differs mode={mode}"


@pytest.mark.parametrize("n,pattern", [(1, "full"), (5, "full"), (1023, "full"), (1025, "full"), (4096, "full"),
                                       (20_000, "full"), (20_000, "ragged"), (100_003, "ragged")])
def test_string_c3_shape(n, pattern):
    dev = _device_mod()
    _check_string(dev, ch.config_c3(n, pattern=pattern, seed=7 + n))


def test_string_golden_and_edge_cases():
    dev = _device_mod()
    rng = np.random.default_rng(5)
    strings = [b"a", None, b"c", None, b"e", b"", b"hello", b"exactly12byt", b"thirteen byte", b"x" * 5000,
               b"embedded\0nul inline", b"in\0l", None, "héllo wörld ✓ utf8".encode(), b"y" * 70000, b""]
    counts = ch.chunk_counts(len(strings))
    _check_string(dev, ch.ChunkBatch(counts, [ch.string_column("s", strings, counts)]))
    # pointer strings scattered in the heap (not in row order)
    many = [None if rng.random() < 0.1 else bytes(rng.integers(1, 255, int(rng.integers(0, 200)), dtype=np.uint8)) for _ in range(5000)]
    counts = ch.chunk_counts(len(many), "ragged", rng)
    _check_string(dev, ch.ChunkBatch(counts, [ch.string_column("s", many, counts, shuffle_heap=rng)]))


def test_string_config_c2_columns():
    dev = _device_mod()
    b = ch.config_c2(30_000)
    for col in range(11, 16):
        _check_string(dev, b, col=col, modes=(0,))


@pytest.mark.parametrize("n,pattern,max_len", [(1, "full", 12), (2048, "full", 1), (2049, "full", 12), (50_000, "ragged", 12),
                                               (70_001, "ragged", 3), (30_000, "full", 0)])
def test_string_inline_only_columns_take_the_whole_vector_kernel(n, pattern, max_len):
    """Columns without a heap (every string inlined), all three modes: the pack kernel's lean form (Arrow modes) and
    string_inline_kernel (reference blob), both on whole-vector tiles."""
    dev = _device_mod()
    rng = np.random.default_rng(900 + n)
    counts = ch.chunk_counts(n, pattern, rng)
    lens = rng.integers(0, max_len + 1, n)
    valid = rng.random(n) > 0.2
    col = ch.string_column_bulk("s", lens, valid, counts, rng, utf8_fraction=0.1)
    assert col.heap.shape[0] <= 16
    _check_string(dev, ch.ChunkBatch(counts, [col]))
    strings = [b"a", None, b"", b"exactly12byt", b"in\0l", b"\0", None, b"xyz"] * 300
    counts = ch.chunk_counts(len(strings))
    _check_string(dev, ch.ChunkBatch(counts, [ch.string_column("s", strings, counts)]))


def test_string_pointer_row_without_a_heap_is_an_error():
    dev = _device_mod()
    strings = [b"short", b"this one is longer than twelve bytes", b"x"]
    counts = ch.chunk_counts(len(strings))
    col = ch.string_column("s", strings, counts)
    col.heap = None  # the batch registers no heap
    db = dev.DeviceBatch(ch.ChunkBatch(counts, [col]))
    so = db.plan_string(0, 0, data_capacity=64)
    db.run_string(so)
    assert db.string_error(so) & 4  # kErrHeapRange


@pytest.mark.parametrize("mode", [0, 2])
def test_string_pointer_outside_the_registered_heap_is_an_error(mode):
    # a string_t whose pointer leaves the registered heap must raise kErrHeapRange (and contribute no bytes),
    # in the Arrow kernels and in the reference-blob kernel
    dev = _device_mod()
    strings = [b"short", b"this one is longer than twelve bytes", b"x", b"another string beyond the inline limit"] * 200
    counts = ch.chunk_counts(len(strings))
    col = ch.string_column("s", strings, counts)
    col.heap = col.heap[: col.heap.shape[0] // 2].copy()  # only the first half of the heap is registered
    db = dev.DeviceBatch(ch.ChunkBatch(counts, [col]))
    so = db.plan_string(0, mode, data_capacity=len(strings) * 64)
    db.run_string(so)
    assert db.string_error(so) & 4  # kErrHeapRange


# ------------------------------------------------------------------ string_pack_kernel paths
def _bulk(n, lens, valid_p, pattern, seed):
    rng = np.random.default_rng(seed)
    counts = ch.chunk_counts(n, pattern, rng)
    valid = None if valid_p is None else rng.random(n) >= valid_p
    return ch.ChunkBatch(counts, [ch.string_column_bulk("s", lens(rng, n), valid, counts, rng, utf8_fraction=0.05)])


@pytest.mark.parametrize("n,pattern", [(513, "full"), (40_000, "full"), (40_000, "ragged")])
def test_string_one_run_tiles(n, pattern):
    # every row a pointer string laid out in row order: each tile is one shifted copy of its heap span;
    # with NULLs (no heap bytes) in between the tiles are still one run
    dev = _device_mod()
    _check_string(dev, _bulk(n, lambda r, m: r.integers(13, 44, m), None, pattern, 11), modes=(0, 1))
    _check_string(dev, _bulk(n, lambda r, m: r.integers(13, 44, m), 0.2, pattern, 12), modes=(0, 1))


@pytest.mark.parametrize("n,pattern", [(3000, "full"), (50_000, "ragged")])
def test_string_few_heap_bytes_per_row(n, pattern):
    # l_shipinstruct shape: a few distinct values around the inline limit -> the 1024-row-tile variant
    dev = _device_mod()
    choices = np.asarray([17, 11, 4, 16, 0, 12, 13])
    _check_string(dev, _bulk(n, lambda r, m: choices[r.integers(0, choices.shape[0], m)], 0.1, pattern, 13))


@pytest.mark.parametrize("tiles", [31, 32, 33, 63, 64, 65, 96, 1025])
@pytest.mark.parametrize("rows_per_tile,lens", [(512, (10, 44)), (1024, None)])
def test_string_pack_lookback_group_boundaries(tiles, rows_per_tile, lens):
    """The pack kernel's two-level look-back reads the <= 63 nearest tiles one by one and everything before them as groups
    of 32 tiles (sum word + prefix word per group): tile counts on both sides of every boundary of that scheme, for the
    512-row-tile kernel (l_comment shape) and the 1024-row-tile kernel (l_shipinstruct shape), int32 and int64 offsets."""
    dev = _device_mod()
    n = rows_per_tile * (tiles - 1) + 7  # the last tile is ragged
    if lens is None:
        choices = np.asarray([17, 11, 4, 16])
        gen = lambda r, m: choices[r.integers(0, 4, m)]  # noqa: E731
    else:
        gen = lambda r, m: r.integers(lens[0], lens[1], m)  # noqa: E731
    _check_string(dev, _bulk(n, gen, 0.05, "full", 500 + tiles), modes=(0, 1))


def test_string_tiles_that_do_not_fit_the_stages():
    # short strings on average (the pack kernel is chosen), but some tiles hold long strings or point all over
    # the heap: those tiles take the row-by-row path inside the same launch
    dev = _device_mod()
    rng = np.random.default_rng(14)
    n = 30_000
    lens = rng.integers(0, 30, n)
    lens[rng.integers(0, n, 12)] = rng.integers(20_000, 70_000, 12)   # a few very long rows
    counts = ch.chunk_counts(n, "ragged", rng)
    col = ch.string_column_bulk("s", lens, rng.random(n) > 0.1, counts, rng)
    _check_string(dev, ch.ChunkBatch(counts, [col]))
    # scattered pointers: reverse the heap order of the pointer strings (every tile's span becomes huge)
    strings = [bytes(rng.integers(0x20, 0x7F, int(l), dtype=np.uint8)) for l in rng.integers(0, 40, 6000)]
    counts = ch.chunk_counts(len(strings))
    col = ch.string_column("s", strings, counts)
    col2 = ch.string_column("s", strings[::-1], counts)   # same strings, heap filled in the opposite order
    # rows in forward order, heap (and pointers) from the reversed column
    data = col2.data.reshape(-1, 16)[: len(strings)][::-1].copy()
    col.data.reshape(-1, 16)[: len(strings)] = data
    col.heap = col2.heap
    _check_string(dev, ch.ChunkBatch(counts, [col]), modes=(0, 1))
