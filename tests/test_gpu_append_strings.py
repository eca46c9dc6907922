"""GPU: Arrow string views (rev_view_kernel) and dictionary-encoded strings (rev_dict_kernel through the string_t table
built once per append) appended to VARCHAR and BLOB columns.

Every case is checked two ways: against tests/reverse_semantics.py (the cells pyarrow's `to_pylist` gives, and the
decoder's vector invariants), and differentially against the same values as plain utf8 / binary appended through the
existing path in the same batch: masks and inline string_t identical, pointer string_t with the same length and prefix
and the same bytes at their targets.  Then the errors and where they stop the append, the positions a VARCHAR / BLOB
column reaches (STRUCT fields under NULL struct rows, LIST children across DMB_REV_LIST_CHILD_CAP cuts), the refusals,
both kernels at the device API, the glue on a mock table, and one 20 M-row append."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
pa = pytest.importorskip("pyarrow")

import reverse_semantics as rs  # noqa: E402
from duckdb_mbt_b200 import chunks as ch  # noqa: E402
from duckdb_mbt_b200 import native as nat  # noqa: E402
from test_rev_enum_cpu import dictionary_array  # noqa: E402
from test_rev_strings_cpu import SUB_ROWS, edge_values, n_for, placed, plain, raw_views, view_array  # noqa: E402

V, B = ch.T_VARCHAR, ch.T_BLOB
INDEX_TYPES = {"c": pa.int8(), "C": pa.uint8(), "s": pa.int16(), "S": pa.uint16(), "i": pa.int32(), "I": pa.uint32(),
               "l": pa.int64(), "L": pa.uint64()}


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


@pytest.fixture(autouse=True)
def _sub_batches(monkeypatch):
    monkeypatch.setenv("DMB_REV_BATCH_ROWS", str(SUB_ROWS))


def _append(ctx, arrays, types, declare=None, **sink_kw):
    from duckdb_mbt_b200 import appender as ap
    batch = pa.StructArray.from_arrays(arrays, names=["c%d" % i for i in range(len(arrays))])
    sink = ap.CollectedChunks(types, **sink_kw)
    a = ap.Appender(ctx, types, sink)
    if declare:
        declare(a)
    a.append_arrow(batch)
    a.flush()
    assert sink.nrows == len(batch)
    a.close()
    return sink


def _same_strings(got_data, got_val, exp_data, exp_val, counts, what):
    """string_t vectors chunk by chunk: masks and inline cells identical, pointer cells with the same len / prefix and the
    same bytes at their targets"""
    for k, cnt in enumerate(counts):
        assert np.array_equal(got_val[k], exp_val[k]), f"{what}: chunk {k} masks"
        g = np.frombuffer(got_data[k], np.uint8).reshape(-1, 16)[:cnt]
        e = np.frombuffer(exp_data[k], np.uint8).reshape(-1, 16)[:cnt]
        lens = g[:, :4].copy().view(np.uint32)[:, 0]
        inline = lens <= 12
        bad = np.nonzero(inline & (g != e).any(axis=1))[0]
        assert not len(bad), f"{what}: chunk {k} row {bad[0]}: {g[bad[0]].tobytes().hex()} vs {e[bad[0]].tobytes().hex()}"
        bad = np.nonzero(~inline & (g[:, :8] != e[:, :8]).any(axis=1))[0]
        assert not len(bad), f"{what}: chunk {k} row {bad[0]}: len / prefix differ"
        gp = g[:, 8:].copy().view(np.uint64)[:, 0]
        ep = e[:, 8:].copy().view(np.uint64)[:, 0]
        for r in np.nonzero(~inline)[0]:
            assert C.string_at(int(gp[r]), int(lens[r])) == C.string_at(int(ep[r]), int(lens[r])), f"{what}: chunk {k} row {r}"


def _check_pair(sink, got_col, exp_col, t, arr, what=""):
    """column got_col (the new encoding of arr) against reverse_semantics and against column exp_col (plain)"""
    assert rs.decode_collected(sink, got_col, t) == rs.expected_cells(arr, t), what
    _same_strings(sink.data[got_col], sink.validity[got_col], sink.data[exp_col], sink.validity[exp_col], sink.counts, what)


# ------------------------------------------------------------------------------------------- views
@pytest.mark.parametrize("binary,off", [(False, k) for k in range(8)] + [(True, 0), (True, 5)])
def test_views_match_the_plain_path(ctx, binary, off):
    rng = np.random.default_rng(off + 10 * binary)
    edges = edge_values()
    n = n_for(edges)
    cells = placed(edges, n, rng)
    full = [b"lead%d" % i if i % 2 else b"leading string number %d" % i for i in range(off)] + cells
    arr = view_array(full, binary=binary, nbufs=3, seed=off).slice(off)
    ref = plain(full, binary).slice(off)
    t = B if binary else V
    sink = _append(ctx, [pa.array(np.arange(n, dtype=np.int32)), arr, ref], [ch.T_INTEGER, t, t])
    _check_pair(sink, 1, 2, t, arr, f"views at offset {off}")


def _corrupt(arr, row, how):
    """a copy of view array `arr` whose view at `row` is malformed"""
    v = raw_views(arr).copy()
    bufs = arr.buffers()
    nbufs = len(bufs) - 2
    x = v[row].view(np.int32)
    assert x[0] > 12
    if how == "index":
        x[2] = nbufs
    elif how == "past-end":
        x[3] = bufs[2 + x[2]].size - x[0] + 1
    elif how == "negative-offset":
        x[3] = -1
    else:
        x[0] = -5
    return pa.Array.from_buffers(arr.type, len(arr), [bufs[0], pa.py_buffer(v.tobytes())] + bufs[2:], null_count=arr.null_count)


WHY = {"index": "buffer index 3 is outside the array's 3 data buffers", "past-end": "pass the end of data buffer",
       "negative-offset": "string view offset -1 is negative", "negative-len": "string view length -5 is negative"}


@pytest.mark.parametrize("how", list(WHY))
def test_malformed_views_stop_the_append_at_their_sub_batch(ctx, how):
    from duckdb_mbt_b200 import appender as ap
    from duckdb_mbt_b200.arrow_result import DuckDBError
    n = 3 * SUB_ROWS + 5
    vals = [b"row %d has a pointer string" % i for i in range(n)]
    bad_row = SUB_ROWS + 1234
    arr = _corrupt(view_array(vals, seed=7), bad_row, how)
    batch = pa.StructArray.from_arrays([pa.array(np.arange(n, dtype=np.int32)), arr], names=["i", "v"])
    sink = ap.CollectedChunks([ch.T_INTEGER, V])
    a = ap.Appender(ctx, [ch.T_INTEGER, V], sink)
    with pytest.raises(DuckDBError) as e:
        a.append_arrow(batch)
    msg = str(e.value)
    assert f"column 1, row {bad_row}: " in msg and WHY[how] in msg, msg
    assert sink.nrows == SUB_ROWS  # the earlier sub-batch reached the sink, the malformed one did not
    a.close()
    # the same view under a NULL row is not read
    valid = np.ones(n, bool)
    valid[bad_row] = False
    masked = pa.Array.from_buffers(arr.type, n, [pa.py_buffer(np.packbits(valid, bitorder="little").tobytes())] + arr.buffers()[1:],
                                   null_count=1)
    ref = plain([None if i == bad_row else v for i, v in enumerate(vals)])  # alive while its pointers are compared
    sink = _append(ctx, [masked, ref], [V, V])
    _check_pair(sink, 0, 1, V, masked, "malformed view under a NULL row")


def test_view_arrays_without_data_buffers(ctx):
    """all-NULL, all-inline and empty view arrays have no data buffers; Arrow C++ exports their (empty) sizes buffer as
    NULL, which is no malformed array: as a column, a LIST child and a dictionary"""
    n = SUB_ROWS + 5
    short = [b"s%d" % (i % 1000) if i % 7 else b"" for i in range(n)]
    views = np.zeros((n, 16), np.uint8)
    for i, v in enumerate(short):
        views[i, :4] = np.frombuffer(np.int32(len(v)).tobytes(), np.uint8)
        views[i, 4:4 + len(v)] = np.frombuffer(v, np.uint8)
    inline = pa.Array.from_buffers(pa.string_view(), n, [None, pa.py_buffer(views.tobytes())])
    assert len(inline.buffers()) == 2
    nulls = pa.array([None] * n, pa.string_view())
    lst = pa.ListArray.from_arrays(pa.array(np.arange(n + 1), pa.int32()), nulls)
    dct = pa.DictionaryArray.from_arrays(pa.array(np.arange(n) % 50, pa.int16()), inline.slice(0, 50))
    arrays = [inline, nulls, lst, dct]
    ref = plain(short)
    sink = _append(ctx, arrays + [ref], [V, V, ch.T_LIST, V, V], declare=lambda a: a.set_list(2, V), list_children={2: (V, 0)})
    _check_pair(sink, 0, 4, V, inline, "all inline")
    assert rs.decode_collected(sink, 1, V) == [None] * n
    assert rs.decode_collected(sink, 2, ch.T_LIST, child=(V, 0)) == [[None]] * n
    assert rs.decode_collected(sink, 3, V) == rs.expected_cells(dct, V)
    empty = [pa.array([], pa.string_view()), pa.array([], pa.string_view()), pa.ListArray.from_arrays(pa.array([0], pa.int32()), nulls.slice(0, 0)),
             pa.DictionaryArray.from_arrays(pa.array([], pa.int16()), inline.slice(0, 0))]
    from duckdb_mbt_b200 import appender as ap
    a = ap.Appender(ctx, [V, V, ch.T_LIST, V], ap.CollectedChunks([V, V, ch.T_LIST, V]))
    a.set_list(2, V)
    a.append_arrow(pa.StructArray.from_arrays(empty, names=["a", "b", "c", "d"]))
    a.flush()
    assert a.row_count == 0
    a.close()


# ------------------------------------------------------------------------------------------- dictionaries
def _dict_case(rng, n, index_fmt, entries, null_frac=0.15):
    """indices over `entries` (a pyarrow array that may hold NULLs); NULL rows carry negative and past-the-end indices;
    every entry appears at the chunk and sub-batch edges"""
    m = len(entries)
    lim = {"c": 127, "s": 32767}.get(index_fmt.lower(), m - 1)
    idx = rng.integers(0, min(m, lim + 1), n).astype(np.int64)
    nulls = rng.random(n) < null_frac
    garbage = np.where(rng.random(n) < 0.5, -1 - rng.integers(0, 3, n), m + rng.integers(0, 3, n))
    if index_fmt in "CSIL":
        garbage = np.abs(garbage) + m
    garbage = np.clip(garbage, -128, {"c": 127, "C": 255}.get(index_fmt, 2**31))
    idx[nulls] = garbage[nulls]
    for r in (0, 2047, 2048, SUB_ROWS - 1, SUB_ROWS, n - 1):
        idx[r], nulls[r] = r % min(m, lim + 1), False
    return dictionary_array(idx, INDEX_TYPES[index_fmt], entries, mask=nulls)


def _entries(binary=False, with_null=True):
    e = edge_values() + [b"label %d, long enough for a pointer" % k for k in range(40)] + [b"s%d" % k for k in range(40)]
    if with_null:
        e = e[:7] + [None] + e[7:]
    return plain(e, binary)


@pytest.mark.parametrize("index_fmt", list(INDEX_TYPES))
def test_dictionaries_match_the_plain_path(ctx, index_fmt):
    rng = np.random.default_rng(ord(index_fmt))
    n = 3 * SUB_ROWS + 77
    entries = _entries()
    arr = _dict_case(rng, n + 5, index_fmt, plain([b"unused"] * 3 + [None if v is None else v.encode() for v in entries.to_pylist()])
                     .slice(3)).slice(5)  # sliced dictionary, sliced indices
    ref = pa.array(arr.to_pylist(), pa.string())
    sink = _append(ctx, [arr, ref], [V, V])
    _check_pair(sink, 0, 1, V, arr, f"dictionary<{index_fmt}>")
    assert sink.valid_bits(0).sum() < n  # NULL rows and NULL entries


@pytest.mark.parametrize("values", ["large_utf8", "binary", "large_binary", "utf8_view", "binary_view"])
def test_dictionary_value_types(ctx, values):
    rng = np.random.default_rng(len(values))
    binary = "binary" in values
    entries = _entries(binary)
    raw = [v if v is None or binary else v.encode() for v in entries.to_pylist()]
    if values.endswith("view"):
        dictionary = view_array(raw, binary=binary, nbufs=2, seed=3)
    else:
        dictionary = entries.cast(pa.large_binary() if binary else pa.large_string()) if values.startswith("large") else entries
    n = 2 * SUB_ROWS + 9
    arr = _dict_case(rng, n, "i", dictionary)
    ref = pa.array(arr.to_pylist(), pa.binary() if binary else pa.string())
    t = B if binary else V
    sink = _append(ctx, [arr, ref], [t, t])
    _check_pair(sink, 0, 1, t, arr, values)


def test_a_dictionary_larger_than_shared_memory(ctx):
    rng = np.random.default_rng(5)
    m = 100_000
    entries = plain([None if k % 997 == 3 else (b"entry number %d" % k if k % 2 else b"e%d" % k) for k in range(m)])
    n = 3 * SUB_ROWS + 1
    arr = dictionary_array(rng.integers(0, m, n), pa.int32(), entries, mask=rng.random(n) < 0.05)
    ref = pa.array(arr.to_pylist(), pa.string())
    sink = _append(ctx, [arr, ref], [V, V])
    _check_pair(sink, 0, 1, V, arr, "100 000 entries")


def test_an_empty_dictionary_with_all_null_rows(ctx):
    n = SUB_ROWS + 3
    arr = dictionary_array(np.arange(n) % 5, pa.int16(), pa.array([], pa.string()), mask=np.ones(n, bool))
    sink = _append(ctx, [arr], [V])
    assert rs.decode_collected(sink, 0, V) == [None] * n


@pytest.mark.parametrize("bad", [-1, "past"])
def test_indices_outside_the_dictionary_stop_the_append(ctx, bad):
    from duckdb_mbt_b200 import appender as ap
    from duckdb_mbt_b200.arrow_result import DuckDBError
    n = 3 * SUB_ROWS
    entries = plain([b"a", b"bb", b"a string of more than twelve bytes"])
    idx = np.arange(n) % 3
    bad_row = 2 * SUB_ROWS + 17
    idx[bad_row] = -1 if bad == -1 else 3
    arr = dictionary_array(idx, pa.int64(), entries)
    sink = ap.CollectedChunks([ch.T_INTEGER, V])
    a = ap.Appender(ctx, [ch.T_INTEGER, V], sink)
    with pytest.raises(DuckDBError) as e:
        a.append_arrow(pa.StructArray.from_arrays([pa.array(np.arange(n, dtype=np.int32)), arr], names=["i", "d"]))
    want = f"column 1, row {bad_row}: dictionary index {idx[bad_row]} is outside the Arrow dictionary (3 entries)"
    assert want in str(e.value), str(e.value)
    assert sink.nrows == 2 * SUB_ROWS
    a.close()


@pytest.mark.parametrize("referenced", [True, False])
def test_a_malformed_view_in_a_view_dictionary_fails_the_append(ctx, referenced):
    """a dictionary of views is converted whole, once per append: a malformed entry fails it before the first sub-batch,
    whether or not a row refers to it"""
    from duckdb_mbt_b200 import appender as ap
    from duckdb_mbt_b200.arrow_result import DuckDBError
    entries = view_array([b"dictionary entry %d, a pointer string" % k for k in range(20)], nbufs=2, seed=9)
    bad = _corrupt(entries, 5, "index")
    n = 2 * SUB_ROWS
    idx = np.arange(n) % 20 if referenced else np.where(np.arange(n) % 20 == 5, 6, np.arange(n) % 20)
    arr = pa.DictionaryArray.from_arrays(pa.array(idx, pa.int32()), bad)
    sink = ap.CollectedChunks([V])
    a = ap.Appender(ctx, [V], sink)
    with pytest.raises(DuckDBError) as e:
        a.append_arrow(pa.StructArray.from_arrays([arr], names=["d"]))
    assert "column 0, dictionary entry 5: string view buffer index 2 is outside the array's 2 data buffers" in str(e.value), str(e.value)
    assert sink.nrows == 0
    a.close()


def test_the_forward_enum_export_appends_into_varchar(ctx):
    from duckdb_mbt_b200 import arrow_result as ar
    rng = np.random.default_rng(11)
    labels = [b"AIR", b"MAIL", b"a label longer than twelve bytes", b""] + [b"label %d" % k for k in range(300)]
    n = 50_000
    counts = ch.chunk_counts(n)
    idx = rng.integers(0, len(labels), n)
    valid = rng.random(n) > 0.1
    col = ch.enum_column("e", labels, idx, counts, valid, garbage_rng=rng)
    res = ar.ArrowResult.from_chunks(ctx, ch.ChunkBatch(counts, [col]))
    arr = res.to_record_batch().column(0)
    assert pa.types.is_dictionary(arr.type)
    ref = pa.array(arr.to_pylist(), pa.string())
    sink = _append(ctx, [arr, ref], [V, V])
    _check_pair(sink, 0, 1, V, arr, "ENUM export")
    assert rs.decode_collected(sink, 0, V) == [labels[i] if ok else None for i, ok in zip(idx, valid)]
    res.close()


# ------------------------------------------------------------------------------------------- positions
def _encodings(rng, n, binary=False):
    """the same n cells as a view array, a dictionary array (NULL entries, out-of-range indices under NULL rows) and plain"""
    vals = placed(edge_values(), n, rng)
    view = view_array(vals, binary=binary, seed=int(rng.integers(1000)))
    entries = _entries(binary)
    dct = _dict_case(rng, n, "s", entries)
    return view, dct


def test_struct_fields_two_deep_under_null_struct_rows(ctx):
    from test_gpu_append_struct import _declare
    rng = np.random.default_rng(21)
    n = 3 * SUB_ROWS + 11
    view, dct = _encodings(rng, n)
    bview, _ = _encodings(rng, n, binary=True)
    outer_null = rng.random(n) < 0.15
    inner_null = rng.random(n) < 0.15
    # out-of-range indices under NULL ancestor rows are not errors
    raw = dct.indices.fill_null(0).to_numpy().astype(np.int64)
    raw[np.nonzero(outer_null)[0][:50]] = 9999
    raw[np.nonzero(inner_null & ~outer_null)[0][:50]] = -7
    dct = dictionary_array(raw, pa.int16(), dct.dictionary, mask=~dct.is_valid().to_numpy(zero_copy_only=False))
    inner = pa.StructArray.from_arrays([dct, bview], names=["d", "b"], mask=pa.array(inner_null))
    outer = pa.StructArray.from_arrays([view, inner], names=["v", "inner"], mask=pa.array(outer_null))
    spec = [("v", V), ("inner", ch.T_STRUCT, [("d", V), ("b", B)])]
    sink = _append(ctx, [outer], [ch.T_STRUCT], declare=lambda a: _declare(a, 0, spec), structs={0: spec})
    rows = sink.struct_values(0)

    def py(v):
        return v.encode() if isinstance(v, str) else v

    exp = outer.to_pylist()
    assert len(rows) == len(exp)
    for i, (g, e) in enumerate(zip(rows, exp)):
        if e is None:
            assert g is None, i
            continue
        ge = {"v": py(g["v"]), "inner": None if g["inner"] is None else {k: py(x) for k, x in g["inner"].items()}}
        ee = {"v": py(e["v"]), "inner": None if e["inner"] is None else {k: py(x) for k, x in e["inner"].items()}}
        assert ge == ee, i
    for key, t in (((0, 0), V), ((0, 1, 0), V), ((0, 1, 1), B)):  # NULL payloads zero, inline padding zero, prefixes
        for k, cnt in enumerate(sink.counts):
            rs.decode_vector(sink.field_data[key][k], bytes(sink.field_validity[key][k].tobytes()), cnt, t)


LIST_CAP = 3000  # DMB_REV_LIST_CHILD_CAP: below a chunk's ~4000 elements, so every chunk is a sub-batch of its own


@pytest.mark.parametrize("kind", ["view", "dictionary"])
def test_list_children_across_child_cap_cuts(ctx, monkeypatch, kind):
    monkeypatch.setenv("DMB_REV_LIST_CHILD_CAP", str(LIST_CAP))
    rng = np.random.default_rng(31)
    n = 4 * 2048 + 5
    lens = rng.integers(0, 4, n)
    off = np.concatenate([[0], np.cumsum(lens)])
    ne = int(off[-1])
    view, dct = _encodings(rng, ne + 2)
    if kind == "dictionary":  # NULL entries on both sides of each chunk boundary's first element
        raw = dct.indices.fill_null(0).to_numpy().astype(np.int64)
        valid = dct.is_valid().to_numpy(zero_copy_only=False)
        null_entry = dct.dictionary.to_pylist().index(None)
        for k in range(1, (n + 2047) // 2048):
            e = int(off[2048 * k]) + 2
            raw[e - 1], raw[e], valid[e - 1], valid[e] = null_entry, null_entry, True, True
        child = dictionary_array(raw, pa.int16(), dct.dictionary, mask=~valid).slice(2)
    else:
        child = view.slice(2)
    lst = pa.ListArray.from_arrays(pa.array(off, pa.int32()), child, mask=pa.array(rng.random(n) < 0.1))
    ref = pa.ListArray.from_arrays(pa.array(off, pa.int32()), pa.array(child.to_pylist(), pa.string()), mask=pa.array(~lst.is_valid().to_numpy(zero_copy_only=False)))
    sink = _append(ctx, [lst, ref], [ch.T_LIST, ch.T_LIST], declare=lambda a: (a.set_list(0, V), a.set_list(1, V)),
                   list_children={0: (V, 0), 1: (V, 0)})
    assert len(sink.counts) == (n + 2047) // 2048
    got = rs.decode_collected(sink, 0, ch.T_LIST, child=(V, 0))
    assert got == rs.expected_lists(lst, V)
    assert got == rs.decode_collected(sink, 1, ch.T_LIST, child=(V, 0))
    for k in range(len(sink.counts)):
        assert np.array_equal(sink.child_validity[0][k], sink.child_validity[1][k]), k


# ------------------------------------------------------------------------------------------- refusals
def _refused(ctx, types, arrays, declare=None) -> str:
    from duckdb_mbt_b200 import appender as ap
    from duckdb_mbt_b200.arrow_result import DuckDBError
    a = ap.Appender(ctx, types, ap.CollectedChunks(types))
    if declare:
        declare(a)
    with pytest.raises(DuckDBError) as e:
        a.append_arrow(pa.StructArray.from_arrays(arrays, names=["c%d" % i for i in range(len(arrays))]))
    a.close()
    return str(e.value)


def test_refusals_name_the_arrow_format(ctx):
    ids = pa.array([1, 2], pa.int32())
    msg = _refused(ctx, [ch.T_INTEGER, V], [ids, pa.array([b"a", None], pa.binary_view())])
    assert "column 1" in msg and "'vz'" in msg, msg
    msg = _refused(ctx, [ch.T_INTEGER, B], [ids, pa.array(["a", None], pa.string_view())])
    assert "column 1" in msg and "'vu'" in msg, msg
    ints = pa.DictionaryArray.from_arrays(pa.array([0, 1], pa.int8()), pa.array([5, 6], pa.int32()))
    msg = _refused(ctx, [ch.T_INTEGER, V], [ids, ints])
    assert "column 1: an Arrow dictionary of 'i' values cannot be appended to a VARCHAR column" in msg, msg
    strs = pa.DictionaryArray.from_arrays(pa.array([0, 1], pa.int8()), pa.array(["x", "y"]))
    msg = _refused(ctx, [ch.T_INTEGER, B], [ids, strs])
    assert "an Arrow dictionary of 'u' values cannot be appended to a BLOB column" in msg, msg
    lst = pa.ListArray.from_arrays(pa.array([0, 1, 2], pa.int32()), ints)
    msg = _refused(ctx, [ch.T_INTEGER, ch.T_LIST], [ids, lst], lambda a: a.set_list(1, V))
    assert "column 1" in msg and "dictionary of 'i' values" in msg, msg


def test_a_view_array_with_fewer_than_three_buffers_is_malformed(ctx):
    from duckdb_mbt_b200 import appender as ap
    batch = pa.StructArray.from_arrays([pa.array(["inline", "a pointer string here"], pa.string_view())], names=["v"])
    a = ap.Appender(ctx, [V], ap.CollectedChunks([V]))
    arr, sch = nat.ArrowArray(), nat.ArrowSchema()
    batch._export_to_c(C.addressof(arr), C.addressof(sch))
    child = arr.children[0].contents
    assert child.n_buffers >= 3
    kept = child.n_buffers
    child.n_buffers = 2
    try:
        ok = a.lib.duckdb_mb_gpu_append_arrow_batch(a.handle, C.addressof(arr), C.addressof(sch))
    finally:
        child.n_buffers = kept
        ap._release(arr)
        ap._release(sch)
    assert not ok
    assert "column 0: the Arrow string view array is malformed: it has 2 buffers" in a.error(), a.error()
    a.close()


# ------------------------------------------------------------------------------------------- L0
def _dev(a: np.ndarray, lead: int = 0):
    t = torch.zeros(lead + a.nbytes + 64, dtype=torch.uint8, device="cuda:0")
    t[lead: lead + a.nbytes] = torch.from_numpy(a.view(np.uint8).reshape(-1).copy()).to("cuda:0")
    return t, t.data_ptr() + lead


def _outputs(n):
    nch = (n + 2047) // 2048
    out = torch.full((nch * 2048 * 16,), 0xAB, dtype=torch.uint8, device="cuda:0")
    val = torch.full((nch * 32,), -1, dtype=torch.int64, device="cuda:0")
    nc = torch.zeros(1, dtype=torch.int64, device="cuda:0")
    err = torch.full((1,), -1, dtype=torch.int64, device="cuda:0")
    return out, val, nc, err


def _expect(cells, valid, n):
    """(string_t rows, mask words) of `cells`: per row None (NULL) or the 16 bytes"""
    nch = (n + 2047) // 2048
    out = np.zeros((nch * 2048, 16), np.uint8)
    bits = np.zeros(nch * 2048, bool)
    for i, c in enumerate(cells):
        if c is not None and valid[i]:
            out[i] = np.frombuffer(c, np.uint8)
            bits[i] = True
    return out, np.packbits(bits, bitorder="little").view(np.uint64)


@pytest.mark.parametrize("n,elem_off,bm_lead", [(1, 0, 1), (2049, 3, 2), (70_001, 7, 3)])
def test_l0_view_kernel(n, elem_off, bm_lead):
    import struct
    L = nat.lib()
    rng = np.random.default_rng(n)
    vals = placed(edge_values(), n + elem_off, rng)
    arr = view_array(vals, nbufs=3, seed=n).slice(elem_off)
    views = raw_views(arr).copy()
    valid = arr.is_valid().to_numpy(zero_copy_only=False)
    bm = np.packbits(np.concatenate([np.zeros(elem_off, bool), valid]), bitorder="little")
    tv, pv = _dev(views)
    tb, pb = _dev(bm, lead=bm_lead)
    bufs = arr.buffers()[2:]
    table = np.asarray([(b.address, b.size) for b in bufs], dtype=np.int64)
    tt, pt = _dev(table)
    out, val, nc, err = _outputs(n)
    job = nat.RevViewJob(pv, pb, elem_off, pt, len(bufs), out.data_ptr(), val.data_ptr(), nc.data_ptr(), err.data_ptr())
    nat.check(L.dmb_dev_rev_view_batch(C.byref(job), n, C.c_void_p(torch.cuda.current_stream().cuda_stream)), "rev_view")
    torch.cuda.synchronize()
    cells = []
    for i in range(n):
        ln = int(views[i, :4].view(np.int32)[0])
        if not valid[i]:  # a NULL row's view is garbage
            cells.append(None)
        elif ln <= 12:
            cells.append(views[i, :4 + ln].tobytes() + bytes(12 - ln))
        else:
            b, o = views[i, 8:16].view(np.int32)
            cells.append(struct.pack("<i4sQ", ln, views[i, 4:8].tobytes(), bufs[b].address + int(o)))
    exp, exp_val = _expect(cells, valid, n)
    got = out.cpu().numpy().reshape(-1, 16)
    assert np.array_equal(got, exp)
    assert np.array_equal(val.cpu().numpy().view(np.uint64), exp_val)
    assert int(nc.item()) == int((~valid).sum())
    assert int(err.item()) == -1


@pytest.mark.parametrize("w", [1, 2, 4, 8])
@pytest.mark.parametrize("n,elem_off,bm_lead,dict_len", [(5, 1, 1, 7), (70_001, 3, 2, 3000), (70_001, 5, 3, 5000)])
def test_l0_dict_kernel(w, n, elem_off, bm_lead, dict_len):
    L = nat.lib()
    rng = np.random.default_rng(n + w + dict_len)
    table = rng.integers(0, 256, (dict_len, 16), dtype=np.uint8)
    null_entries = rng.random(dict_len) < 0.1
    table.view(np.uint32)[null_entries, 0] = nat.DICT_ENTRY_NULL
    dt = {1: np.int8, 2: np.int16, 4: np.int32, 8: np.int64}[w]
    hi = min(dict_len, np.iinfo(dt).max + 1)
    idx = rng.integers(0, hi, n + elem_off).astype(dt)
    bm = rng.integers(0, 256, (n + elem_off + 7) // 8 + 1, dtype=np.uint8)
    valid = np.unpackbits(bm, bitorder="little")[elem_off:elem_off + n].astype(bool)
    bad = np.nonzero(valid)[0][-1]
    idx[elem_off + bad] = -1  # the one error; out-of-range indices under NULL rows are not errors
    idx[elem_off + np.nonzero(~valid)[0][:5]] = -3
    ti, pi = _dev(idx)
    tb, pb = _dev(bm, lead=bm_lead)
    tt, pt = _dev(table)
    out, val, nc, err = _outputs(n)
    job = nat.RevDictJob(pi + elem_off * w, pb, elem_off, pt, dict_len, out.data_ptr(), val.data_ptr(), nc.data_ptr(), err.data_ptr(), w, 1)
    nat.check(L.dmb_dev_rev_dict_batch(C.byref(job), n, C.c_void_p(torch.cuda.current_stream().cuda_stream)), "rev_dict")
    torch.cuda.synchronize()
    ix = idx[elem_off:].astype(np.int64)
    ok = valid & (ix >= 0) & (ix < dict_len)
    ok[ok] &= ~null_entries[ix[ok]]
    cells = [table[ix[i]].tobytes() if ok[i] else None for i in range(n)]
    exp, exp_val = _expect(cells, ok, n)
    assert np.array_equal(out.cpu().numpy().reshape(-1, 16), exp)
    assert np.array_equal(val.cpu().numpy().view(np.uint64), exp_val)
    assert int(nc.item()) == int(n - ok.sum())
    assert int(err.item()) == bad


# ------------------------------------------------------------------------------------------- glue + mock DuckDB
def test_glue_appends_views_and_dictionaries():
    """A mock table of VARCHAR, BLOB and STRUCT{VARCHAR}: a view column, a dictionary column and a dictionary field go
    through glue/duckdb_gpu_glue.c, which copies each string into the table; read back, the table holds the plain cells."""
    from test_glue_mock import Glue
    from test_gpu_append_struct import _mock_read
    from duckdb_mbt_b200 import appender as ap
    g = Glue()
    vp, i32p = C.c_void_p, C.POINTER(C.c_int32)
    g.mock.duckdb_mock_set_append_struct.argtypes = [C.c_char_p, C.c_int32, i32p, C.c_int32, C.c_int32, i32p, i32p, i32p]
    g.mock.duckdb_mock_appended_struct_field.restype = C.c_int64
    g.mock.duckdb_mock_appended_struct_field.argtypes = [C.c_char_p, C.c_int64, C.c_int32, i32p, C.c_int32, C.POINTER(vp), C.POINTER(vp)]
    table = b"t_strings"
    types = np.asarray([V, B, ch.T_STRUCT], dtype=np.int32)
    assert g.mock.duckdb_mock_register_append_table(b"main", table, 3, types.ctypes.data, None, None)
    assert g.mock.duckdb_mock_set_append_struct(table, 2, None, 0, 1, (C.c_int32 * 1)(V), None, None)
    h = g.glue.duckdb_mb_appender_create(C.byref(g.conn), g.bytes_(b"main"), g.bytes_(table))
    assert h
    rng = np.random.default_rng(41)
    n = 5000
    view, dct = _encodings(rng, n)
    _, bdct = _encodings(rng, n, binary=True)
    st = pa.StructArray.from_arrays([dct], names=["d"], mask=pa.array(rng.random(n) < 0.2))
    batch = pa.StructArray.from_arrays([view, bdct, st], names=["v", "b", "s"])
    L = nat.lib()
    arr, sch = nat.ArrowArray(), nat.ArrowSchema()
    batch._export_to_c(C.addressof(arr), C.addressof(sch))
    try:
        ok = L.duckdb_mb_gpu_append_arrow_batch(vp(h), C.addressof(arr), C.addressof(sch))
    finally:
        ap._release(arr)
        ap._release(sch)
    assert ok, nat.moonbit_bytes(L.duckdb_mb_gpu_appender_error(vp(h)))
    assert L.duckdb_mb_gpu_appender_flush(vp(h))
    nch = g.mock.duckdb_mock_appended_chunks(table)
    assert nch == 3
    for col, t, a in ((0, V, view), (1, B, bdct)):
        got = []
        for k in range(nch):
            d, m = vp(), vp()
            cnt = g.mock.duckdb_mock_appended_chunk(table, k, col, C.byref(d), C.byref(m))
            got += rs.decode_vector(C.string_at(d.value, 16 * cnt), C.string_at(m.value, 256) if m.value else None, cnt, t, strict=False)
        assert got == rs.expected_cells(a, t), col
    svalid = st.is_valid().to_numpy(zero_copy_only=False)
    got = []
    for k in range(nch):
        cnt, d, m = _mock_read(g, table, k, 2, [0])
        got += rs.decode_vector(C.string_at(d, 16 * cnt), C.string_at(m, 256) if m else None, cnt, V, strict=False)
    assert got == [c if ok else None for c, ok in zip(rs.expected_cells(dct, V), svalid)]
    L.duckdb_mb_appender_destroy.argtypes = [vp]
    L.duckdb_mb_appender_destroy(vp(h))


# ------------------------------------------------------------------------------------------- scale
def test_twenty_million_rows(ctx, monkeypatch):
    """one 20 M-row append of a view column and a dictionary column, at the default sub-batch size; checked with numpy"""
    from duckdb_mbt_b200 import appender as ap
    monkeypatch.delenv("DMB_REV_BATCH_ROWS")
    n = 20_000_000
    rng = np.random.default_rng(51)
    lens = rng.integers(0, 40, n).astype(np.int32)
    data = rng.integers(97, 123, int(lens.sum()) + 16, dtype=np.uint8)
    offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    views = np.zeros((n, 4), np.int32)
    views[:, 0] = lens
    inline = lens <= 12
    vb = views.view(np.uint8).reshape(n, 16)
    for r0 in range(0, n, 1 << 20):  # inline views: their bytes zero-padded; pointer views: prefix, buffer 0, offset
        r1 = min(n, r0 + (1 << 20))
        b12 = data[offs[r0:r1, None] + np.arange(12)[None, :]]
        b12[np.arange(12)[None, :] >= lens[r0:r1, None]] = 0
        vb[r0:r1, 4:16] = b12
    views[~inline, 2] = 0
    views[~inline, 3] = offs[:-1][~inline].astype(np.int32)
    valid = rng.random(n) > 0.05
    bm = pa.py_buffer(np.packbits(valid, bitorder="little").tobytes())
    view = pa.Array.from_buffers(pa.string_view(), n, [bm, pa.py_buffer(views.tobytes()), pa.py_buffer(data.tobytes())],
                                 null_count=int((~valid).sum()))
    m = 70_000
    entries = plain([b"dictionary entry %d" % k if k % 3 else b"e%d" % k for k in range(m)])
    idx = rng.integers(0, m, n).astype(np.int32)
    dct = pa.DictionaryArray.from_arrays(pa.array(idx, mask=~valid), entries)
    sink = ap.CollectedChunks([V, V])
    a = ap.Appender(ctx, [V, V], sink)
    a.append_arrow(pa.StructArray.from_arrays([view, dct], names=["v", "d"]))
    a.flush()
    a.close()
    assert sink.nrows == n
    assert np.array_equal(sink.valid_bits(0), valid) and np.array_equal(sink.valid_bits(1), valid)
    got = np.frombuffer(sink.column_bytes(0), np.uint8).reshape(n, 16)
    exp = np.where(valid[:, None], vb, 0).astype(np.uint8)
    exp_ptr = view.buffers()[2].address + offs[:-1]
    ptr_rows = valid & ~inline
    assert np.array_equal(got[~ptr_rows], exp[~ptr_rows])
    assert np.array_equal(got[ptr_rows, :8], exp[ptr_rows, :8])
    assert np.array_equal(got[ptr_rows, 8:].copy().view(np.uint64)[:, 0], exp_ptr[ptr_rows].astype(np.uint64))
    d = np.frombuffer(sink.column_bytes(1), np.uint8).reshape(n, 16)
    dl = d[:, :4].copy().view(np.uint32)[:, 0]
    elen = np.asarray([len(e) for e in entries.to_pylist()], np.uint32)[idx]
    assert np.array_equal(dl, np.where(valid, elen, 0))
    for r in rng.integers(0, n, 2000):  # spot checks of the bytes
        if valid[r]:
            assert rs.decode_cell(d[r].tobytes(), V) == entries[int(idx[r])].as_py().encode()
