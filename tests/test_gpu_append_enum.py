"""GPU: Arrow dictionary arrays and utf8 labels appended to DuckDB ENUM columns (rev_enum_index_kernel through the remap
the lookup kernel builds from the Arrow dictionary, rev_enum_string_kernel for plain labels), checked against the
reference of tests/test_rev_enum_cpu.py: positions, masks, zero payloads under NULL rows, the errors and where they stop
the append, the refusals, the forward -> reverse round trip, the row protocol and the glue on a mock table."""
import ctypes as C
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
pa = pytest.importorskip("pyarrow")

from duckdb_mbt_b200 import chunks as ch  # noqa: E402
from duckdb_mbt_b200 import native as nat  # noqa: E402
from test_rev_enum_cpu import dictionary_array, enum_reference  # noqa: E402

U8, U16, U32 = ch.T_UTINYINT, ch.T_USMALLINT, ch.T_UINTEGER
INDEX_TYPES = {"c": pa.int8(), "C": pa.uint8(), "s": pa.int16(), "S": pa.uint16(), "i": pa.int32(), "I": pa.uint32(),
               "l": pa.int64(), "L": pa.uint64()}
MAX_INDEX = {"c": 127, "C": 255, "s": 32767, "S": 65535, "i": 2**31 - 1, "I": 2**32 - 1, "l": 2**63 - 1, "L": 2**64 - 1}


@pytest.fixture(autouse=True)
def _needs_device():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


@pytest.fixture(scope="module")
def ctx():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from duckdb_mbt_b200 import arrow_result as ar
    c = ar.GpuContext(0)
    yield c
    c.close()


@functools.lru_cache(maxsize=None)
def _cached_labels(n):
    return make_labels(n, np.random.default_rng(n))


def make_labels(n, rng, lens=(1, 24)):
    """n distinct str labels of lens[0]..lens[1] characters"""
    out, seen = [], set()
    while len(out) < n:
        s = "".join(chr(c) for c in rng.integers(97, 123, int(rng.integers(lens[0], lens[1] + 1))))
        s = s + str(len(out)) if s in seen else s
        if s not in seen:
            seen.add(s)
            out.append(s)
    return out


def _append(ctx, arrays, type_ids, enums):
    """append a record batch of `arrays`; enums {col: (internal_type, labels)}; returns the sink"""
    from duckdb_mbt_b200 import appender as ap
    rb = pa.record_batch(arrays, names=["c%d" % i for i in range(len(arrays))])
    sink = ap.CollectedChunks(type_ids, enums=enums)
    a = ap.Appender(ctx, type_ids, sink)
    for c, (it, labels) in enums.items():
        a.set_enum(c, labels, it)
    a.append_arrow(rb)
    a.flush()
    assert a.state == ap.FLUSHED and sink.nrows == len(rb)
    a.close()
    return sink


def _check(sink, c, arr, labels):
    pos, valid, first = enum_reference(arr, labels)
    assert first is None
    got = sink.enum_positions(c)
    assert np.array_equal(sink.valid_bits(c), valid)
    assert np.array_equal(got, np.where(valid, pos, 0).astype(got.dtype))  # NULL payloads are zero
    for k, cnt in enumerate(sink.counts):  # mask bits past the chunk's count are zero
        bits = np.unpackbits(sink.validity[c][k].view(np.uint8), bitorder="little")
        assert not bits[cnt:].any()


def _dictionary_case(labels, index_fmt, large, rng, n, with_null_entry=True):
    """an Arrow dictionary array over `labels`: the dictionary is shuffled, holds a subset of the labels that fits the index
    type plus an unused non-label and a NULL entry; NULL rows carry negative and out-of-range indices"""
    cap = min(MAX_INDEX[index_fmt] + 1, len(labels) + 2)
    take = rng.permutation(len(labels))[: cap - 2]
    entries = [labels[i] for i in take] + ["not an enum label"] + ([None] if with_null_entry else [])
    order = rng.permutation(len(entries))
    entries = [entries[i] for i in order]
    unused = entries.index("not an enum label")
    usable = np.asarray([i for i in range(len(entries)) if i != unused])
    idx = usable[rng.integers(0, len(usable), n)].astype(np.int64)
    nulls = rng.random(n) < 0.15
    garbage = rng.integers(-3, 3, n) + np.where(rng.random(n) < 0.5, 0, len(entries))
    if index_fmt in "CSIL":
        garbage = np.abs(garbage) + len(entries)
    garbage = np.clip(garbage, -128, MAX_INDEX[index_fmt])
    idx[nulls] = garbage[nulls]
    for r in (0, 2047, 2048, 4095, 4096, n - 1):  # chunk and sub-batch edges, the last row
        idx[r], nulls[r] = usable[-1], False
    dictionary = pa.array(entries, pa.large_string() if large else pa.string())
    return dictionary_array(idx, INDEX_TYPES[index_fmt], dictionary, mask=nulls)


@pytest.mark.parametrize("internal,nlabels", [(U8, 3), (U8, 256), (U16, 300), (U32, 70_000)])
@pytest.mark.parametrize("large", [False, True])
@pytest.mark.parametrize("index_fmt", list(INDEX_TYPES))
def test_dictionary_arrays(ctx, monkeypatch, index_fmt, large, internal, nlabels):
    monkeypatch.setenv("DMB_REV_BATCH_ROWS", "4096")
    rng = np.random.default_rng(nlabels + ord(index_fmt))
    labels = list(_cached_labels(nlabels))
    n = 10_003
    arr = _dictionary_case(labels, index_fmt, large, rng, n)
    ids = pa.array(np.arange(n, dtype=np.int32))
    sink = _append(ctx, [ids, arr], [ch.T_INTEGER, ch.T_ENUM], {1: (internal, labels)})
    _check(sink, 1, arr, labels)
    assert sink.column_bytes(0) == np.arange(n, dtype=np.int32).tobytes()


@pytest.mark.parametrize("offset", range(8))
def test_dictionary_arrays_at_every_offset_with_a_sliced_dictionary(ctx, offset):
    rng = np.random.default_rng(offset)
    labels = make_labels(40, rng)
    arr = _dictionary_case(labels, "S", False, rng, 5000 + offset)
    d = arr.dictionary
    shifted = pa.concat_arrays([pa.array(["x", "y", "z"]), d]).slice(3)  # a dictionary with its own offset
    arr = pa.DictionaryArray.from_arrays(arr.indices, shifted, safe=False).slice(offset)
    sink = _append(ctx, [arr], [ch.T_ENUM], {0: (U8, labels)})
    _check(sink, 0, arr, labels)


EDGE_LABELS = ["", "a", "ab", "abc", "x" * 12, "x" * 13, "a" + "é" * 6, "ab\x00cd", "pre", "prefix", "prefix_0000_mid_tail",
               "prefix_0000_MID_tail", "日本語のラベル・長い", "z" * 70_000]


@pytest.mark.parametrize("large", [False, True])
def test_string_labels(ctx, monkeypatch, large):
    monkeypatch.setenv("DMB_REV_BATCH_ROWS", "4096")
    rng = np.random.default_rng(3)
    n = 9001
    pick = rng.integers(0, len(EDGE_LABELS), n)
    vals = [None if rng.random() < 0.1 else EDGE_LABELS[p] for p in pick]
    for r, p in ((0, 0), (2047, 13), (2048, 7), (4095, 12), (4096, 5), (n - 1, 6)):
        vals[r] = EDGE_LABELS[p]
    arr = pa.array(vals, pa.large_string() if large else pa.string()).slice(1)
    sink = _append(ctx, [arr], [ch.T_ENUM], {0: (U8, EDGE_LABELS)})
    _check(sink, 0, arr, EDGE_LABELS)


def test_every_label_of_a_large_enum_in_shuffled_order(ctx):
    rng = np.random.default_rng(70)
    labels = make_labels(70_000, rng, (1, 30))
    order = rng.permutation(len(labels))
    arr = pa.array([labels[i] for i in order])
    sink = _append(ctx, [arr], [ch.T_ENUM], {0: (U32, labels)})
    assert np.array_equal(sink.enum_positions(0), order.astype(np.uint32))
    assert sink.valid_bits(0).all()


# ------------------------------------------------------------------------------------------- errors and refusals
def _failing(ctx, arrays, type_ids, enums, sink=None, declare=True):
    from duckdb_mbt_b200 import appender as ap
    from duckdb_mbt_b200.arrow_result import DuckDBError
    rb = pa.record_batch(arrays, names=["c%d" % i for i in range(len(arrays))])
    a = ap.Appender(ctx, type_ids, sink or ap.CollectedChunks(type_ids, enums=enums))
    if declare:
        for c, (it, labels) in enums.items():
            a.set_enum(c, labels, it)
    with pytest.raises(DuckDBError) as e:
        a.append_arrow(rb)
    assert a.state == ap.ERROR
    a.close()
    return str(e.value)


def test_a_missing_label_stops_before_its_sub_batch(ctx, monkeypatch):
    from duckdb_mbt_b200 import appender as ap
    monkeypatch.setenv("DMB_REV_BATCH_ROWS", "4096")
    labels = ["AIR", "MAIL", "SHIP"]
    vals = [labels[i % 3] for i in range(20_000)]
    vals[10_001] = "RAIL"
    vals[10_500] = "TRUCK"
    sink = ap.CollectedChunks([ch.T_ENUM], enums={0: (U8, labels)})
    msg = _failing(ctx, [pa.array(vals)], [ch.T_ENUM], {0: (U8, labels)}, sink)
    assert "column 0" in msg and "row 10001" in msg and "'RAIL'" in msg
    assert sink.nrows == 8192  # sub-batches 0 and 1 reached the sink


def test_an_out_of_range_index_stops_before_its_sub_batch(ctx, monkeypatch):
    from duckdb_mbt_b200 import appender as ap
    monkeypatch.setenv("DMB_REV_BATCH_ROWS", "4096")
    labels = ["AIR", "MAIL", "SHIP"]
    idx = np.arange(20_000) % 3
    idx[9000] = 3
    arr = dictionary_array(idx, pa.int32(), pa.array(labels))
    sink = ap.CollectedChunks([ch.T_INTEGER, ch.T_ENUM], enums={1: (U8, labels)})
    msg = _failing(ctx, [pa.array(np.arange(20_000, dtype=np.int32)), arr], [ch.T_INTEGER, ch.T_ENUM], {1: (U8, labels)}, sink)
    assert "column 1" in msg and "row 9000" in msg and "index 3" in msg
    assert sink.nrows == 8192
    arr = dictionary_array([0, 1, 2], pa.int8(), pa.array(["AIR", "RAIL", "SHIP"]))
    assert "row 1" in _failing(ctx, [arr], [ch.T_ENUM], {0: (U8, labels)}) and "'RAIL'" in _failing(ctx, [arr], [ch.T_ENUM], {0: (U8, labels)})


def test_long_labels_are_cut_in_the_message(ctx):
    msg = _failing(ctx, [pa.array(["q" * 5000])], [ch.T_ENUM], {0: (U8, ["a"])})
    assert "row 0" in msg and "..." in msg and len(msg) < 256


def test_refusals(ctx):
    from duckdb_mbt_b200 import appender as ap
    from duckdb_mbt_b200.arrow_result import DuckDBError
    e = {0: (U8, ["a", "b"])}
    assert "duckdb_mb_gpu_appender_set_enum" in _failing(ctx, [pa.array(["a"])], [ch.T_ENUM], e, declare=False)
    assert "bare Arrow integer array" in _failing(ctx, [pa.array([0, 1], pa.uint8())], [ch.T_ENUM], e)
    assert "dictionary of 'l' values" in _failing(ctx, [pa.DictionaryArray.from_arrays(pa.array([0], pa.int8()), pa.array([5]))], [ch.T_ENUM], e)
    if hasattr(pa, "string_view"):
        assert "string views" in _failing(ctx, [pa.array(["a"], pa.string_view())], [ch.T_ENUM], e)
    a = ap.Appender(ctx, [ch.T_ENUM, ch.T_INTEGER, ch.T_LIST], ap.CollectedChunks([ch.T_ENUM, ch.T_INTEGER, ch.T_LIST], enums=e))
    with pytest.raises(DuckDBError, match="has no declared labels"):
        a.begin_row()
    a.close()
    a = ap.Appender(ctx, [ch.T_ENUM, ch.T_INTEGER, ch.T_LIST], ap.CollectedChunks([ch.T_ENUM, ch.T_INTEGER, ch.T_LIST], enums=e))
    with pytest.raises(DuckDBError, match="not an ENUM column"):
        a.set_enum(1, ["a"], U8)
    with pytest.raises(DuckDBError, match="not UTINYINT, USMALLINT or UINTEGER"):
        a.set_enum(0, ["a"], ch.T_BIGINT)
    with pytest.raises(DuckDBError, match="more than internal type"):
        a.set_enum(0, ["l%d" % i for i in range(257)], U8)
    with pytest.raises(DuckDBError, match="both 'b'"):
        a.set_enum(0, ["a", "b", "b"], U8)
    d = nat.EnumDict(2, 0, np.asarray([0, 3, 1], np.uint32).ctypes.data, C.cast(C.c_char_p(b"abc"), C.c_void_p))
    assert not a.lib.duckdb_mb_gpu_appender_set_enum(a.handle, 0, U8, C.byref(d))
    assert "malformed offsets" in a.error()
    a.set_enum(0, ["a", "b"], U8)
    a.set_enum(0, ["a", "b"], U8)  # the same declaration again is fine
    with pytest.raises(DuckDBError, match="different ENUM declaration"):
        a.set_enum(0, ["a", "c"], U8)
    with pytest.raises(DuckDBError, match="LIST child type 23"):
        a.set_list(2, ch.T_ENUM)
    a.close()


# ------------------------------------------------------------------------------------------- round trip
@pytest.mark.parametrize("nlabels,label_len", [(7, (3, 10)), (300, (8, 24))])  # the fused and the two-step forward forms
def test_forward_export_then_append_round_trips(ctx, nlabels, label_len):
    from duckdb_mbt_b200 import arrow_result as ar
    rng = np.random.default_rng(nlabels)
    labels = make_labels(nlabels, rng, label_len)
    n = 50_000
    counts = ch.chunk_counts(n)
    idx = rng.integers(0, nlabels, n)
    valid = rng.random(n) > 0.1
    col = ch.enum_column("e", [x.encode() for x in labels], idx, counts, valid, garbage_rng=rng)
    res = ar.ArrowResult.from_chunks(ctx, ch.ChunkBatch(counts, [col]))
    rb = res.to_record_batch()
    assert pa.types.is_dictionary(rb.column(0).type)
    internal = U8 if nlabels <= 256 else U16
    sink = _append(ctx, [rb.column(0)], [ch.T_ENUM], {0: (internal, labels)})
    res.close()
    dt = np.uint8 if nlabels <= 256 else np.uint16
    src = col.data.view(dt)[:n]
    assert np.array_equal(sink.valid_bits(0), valid)
    assert np.array_equal(sink.enum_positions(0), np.where(valid, src, 0).astype(dt))


# ------------------------------------------------------------------------------------------- row protocol
def test_row_protocol_appends_labels(ctx):
    from duckdb_mbt_b200 import appender as ap
    from duckdb_mbt_b200.arrow_result import DuckDBError
    labels = ["", "AIR", "x" * 20]
    enums = {1: (U16, labels)}
    sink = ap.CollectedChunks([ch.T_INTEGER, ch.T_ENUM], enums=enums)
    a = ap.Appender(ctx, [ch.T_INTEGER, ch.T_ENUM], sink)
    a.set_enum(1, labels, U16)
    want = []
    for i in range(5000):
        a.begin_row()
        a.append_int(i)
        if i % 7 == 3:
            a.append_null()
            want.append(None)
        else:
            a.append_varchar(labels[i % 3])
            want.append(labels[i % 3])
        a.end_row()
    a.flush()
    assert sink.enum_values(1) == want
    assert np.array_equal(sink.enum_positions(1)[np.asarray([w is None for w in want])], np.zeros(sum(w is None for w in want), np.uint16))
    a.begin_row()
    a.append_int(1)
    a.append_varchar("RAIL")
    a.end_row()
    with pytest.raises(DuckDBError, match="'RAIL' is not a label"):
        a.flush()
    assert a.state == ap.ERROR
    a.close()
    for bad in ("append_int", "append_blob"):
        a = ap.Appender(ctx, [ch.T_ENUM], ap.CollectedChunks([ch.T_ENUM], enums={0: (U8, labels)}))
        a.set_enum(0, labels, U8)
        a.begin_row()
        with pytest.raises(DuckDBError, match="has DuckDB type 23"):
            getattr(a, bad)(1 if bad == "append_int" else b"AIR")
        assert a.state == ap.ERROR
        a.close()


# ------------------------------------------------------------------------------------------- glue + mock DuckDB
@pytest.mark.parametrize("width", [1, 2])
def test_glue_appends_enum_columns(width):
    from test_glue_mock import Glue
    from duckdb_mbt_b200 import appender as ap
    g = Glue()
    vp = C.c_void_p
    g.mock.duckdb_mock_set_append_enum.argtypes = [C.c_char_p, C.c_int32, C.c_int32, C.c_uint32, vp]
    rng = np.random.default_rng(width)
    labels = make_labels(5 if width == 1 else 1000, rng)
    table = b"t_enum%d" % width
    types = np.asarray([ch.T_INTEGER, ch.T_ENUM], dtype=np.int32)
    assert g.mock.duckdb_mock_register_append_table(b"main", table, 2, types.ctypes.data, None, None)
    bufs = [C.create_string_buffer(x.encode()) for x in labels]
    ptrs = (C.c_char_p * len(bufs))(*[C.cast(b, C.c_char_p) for b in bufs])
    assert g.mock.duckdb_mock_set_append_enum(table, 1, width, len(labels), C.cast(ptrs, vp))
    h = g.glue.duckdb_mb_appender_create(C.byref(g.conn), g.bytes_(b"main"), g.bytes_(table))
    assert h
    L = nat.lib()
    n = 5000
    dict_arr = _dictionary_case(labels, "i", False, rng, n)
    str_arr = pa.array([None if i % 11 == 0 else labels[int(rng.integers(0, len(labels)))] for i in range(n)])
    want = []
    for arr in (dict_arr, str_arr):
        struct = pa.record_batch([pa.array(np.arange(n, dtype=np.int32)), arr], names=["i", "e"]).to_struct_array()
        a, s = nat.ArrowArray(), nat.ArrowSchema()
        struct._export_to_c(C.addressof(a), C.addressof(s))
        try:
            ok = L.duckdb_mb_gpu_append_arrow_batch(vp(h), C.addressof(a), C.addressof(s))
        finally:
            ap._release(a)
            ap._release(s)
        assert ok, nat.moonbit_bytes(L.duckdb_mb_gpu_appender_error(vp(h)))
        pos, valid, _ = enum_reference(arr, labels)
        want += [int(p) if v else None for p, v in zip(pos, valid)]
    for name, at in (("duckdb_mb_begin_row", [vp]), ("duckdb_mb_append_int", [vp, C.c_int32]), ("duckdb_mb_append_varchar", [vp, vp]),
                     ("duckdb_mb_append_null", [vp]), ("duckdb_mb_end_row", [vp])):
        getattr(L, name).argtypes = at
    for i in range(300):
        assert L.duckdb_mb_begin_row(vp(h)) and L.duckdb_mb_append_int(vp(h), i)
        if i % 5 == 0:
            assert L.duckdb_mb_append_null(vp(h))
            want.append(None)
        else:
            assert L.duckdb_mb_append_varchar(vp(h), g.bytes_(labels[i % len(labels)].encode()))
            want.append(i % len(labels))
        assert L.duckdb_mb_end_row(vp(h))
    assert L.duckdb_mb_gpu_appender_flush(vp(h)), nat.moonbit_bytes(L.duckdb_mb_gpu_appender_error(vp(h)))
    got = []
    dt = np.uint8 if width == 1 else np.uint16
    for k in range(g.mock.duckdb_mock_appended_chunks(table)):
        dptr, mptr = vp(), vp()
        cnt = g.mock.duckdb_mock_appended_chunk(table, k, 1, C.byref(dptr), C.byref(mptr))
        vals = np.frombuffer(C.string_at(dptr.value, cnt * width), dtype=dt)
        valid = (np.unpackbits(np.frombuffer(C.string_at(mptr.value, 256), dtype=np.uint8), bitorder="little")[:cnt].astype(bool)
                 if mptr.value else np.ones(cnt, bool))
        assert not vals[~valid].any()
        got += [int(v) if ok else None for v, ok in zip(vals, valid)]
    assert got == want
    L.duckdb_mb_appender_destroy.argtypes = [vp]
    L.duckdb_mb_appender_destroy(vp(h))


# ------------------------------------------------------------------------------------------- scale
def test_twenty_million_rows_per_path(ctx):
    rng = np.random.default_rng(20)
    labels = make_labels(10_000, rng, (8, 24))
    n = 20_000_000
    # dictionary path: a shuffled Arrow dictionary of every label; numpy restatement = take through the remap
    perm = rng.permutation(len(labels))
    idx = rng.integers(0, len(labels), n).astype(np.int32)
    valid = rng.random(n) > 0.05
    arr = pa.DictionaryArray.from_arrays(pa.array(idx, mask=~valid), pa.array([labels[p] for p in perm]))
    sink = _append(ctx, [arr], [ch.T_ENUM], {0: (U16, labels)})
    assert np.array_equal(sink.valid_bits(0), valid)
    assert np.array_equal(sink.enum_positions(0), np.where(valid, perm.astype(np.uint16)[idx], 0).astype(np.uint16))
    # string path: the same rows as utf8 labels
    del sink
    sarr = arr.cast(pa.string())
    sink = _append(ctx, [sarr], [ch.T_ENUM], {0: (U16, labels)})
    assert np.array_equal(sink.valid_bits(0), valid)
    assert np.array_equal(sink.enum_positions(0), np.where(valid, perm.astype(np.uint16)[idx], 0).astype(np.uint16))
