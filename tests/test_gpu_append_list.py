"""GPU: Arrow list / large_list columns appended to DuckDB LIST columns (rev_list_kernel + the child range converted as a
dense column).  L0 against the numpy restatement of tests/test_rev_list_cpu.py; L1 through Appender.append_arrow against
pyarrow's `to_pylist`; a forward -> reverse round trip of tests/list_cases.py columns; the refusals; and the glue
(duckdb_mb_appender_create on a mock table) filling the LIST vectors' child vectors."""
import ctypes as C
import decimal

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
pa = pytest.importorskip("pyarrow")

from duckdb_mbt_b200 import chunks as ch  # noqa: E402
from duckdb_mbt_b200 import native as nat  # noqa: E402
from test_rev_list_cpu import arrow_parts, make_list_array, rev_list_reference  # noqa: E402


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


# ------------------------------------------------------------------------------------------- L0
def _dev(buf: bytes, pad: int = 64):
    t = torch.zeros(len(buf) + pad, dtype=torch.uint8, device="cuda:0")
    if len(buf):
        t[: len(buf)] = torch.frombuffer(bytearray(buf), dtype=torch.uint8).to("cuda:0")
    return t


def _run_list(off_bytes: bytes, large: bool, n: int, bm: bytes, bit_off: int, cbm: bytes, cbit_off: int, cword: np.ndarray):
    """one dmb_dev_rev_list_batch launch on device copies; returns (entries, masks, child masks, null count, error)"""
    L = nat.lib()
    nch = (n + 2047) // 2048
    keep = [_dev(off_bytes)]
    pb = pc = None
    if bm is not None:
        keep.append(_dev(bm))
        pb = keep[-1].data_ptr()
    if cbm is not None:
        keep.append(_dev(cbm))
        pc = keep[-1].data_ptr()
    cw = torch.from_numpy(cword.astype(np.int64)).to("cuda:0")
    ent = torch.full((nch * 2048 * 16,), 0xAB, dtype=torch.uint8, device="cuda:0")
    val = torch.full((nch * 32,), -1, dtype=torch.int64, device="cuda:0")
    cval = torch.full((int(cword[-1]) + 1,), -1, dtype=torch.int64, device="cuda:0")
    nc = torch.zeros(1, dtype=torch.int64, device="cuda:0")
    err = torch.zeros(1, dtype=torch.int32, device="cuda:0")
    job = nat.RevListJob(keep[0].data_ptr(), pb, bit_off, pc, cbit_off, cw.data_ptr(), ent.data_ptr(), val.data_ptr(), cval.data_ptr(),
                         nc.data_ptr(), err.data_ptr(), 1 if large else 0, 0)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    nat.check(L.dmb_dev_rev_list_batch(C.byref(job), n, st), "rev_list")
    torch.cuda.synchronize()
    return (ent.cpu().numpy().view(np.uint64).reshape(-1, 2), val.cpu().numpy().view(np.uint64),
            cval.cpu().numpy().view(np.uint64), int(nc.item()), int(err.item()))


def _check_l0(arr):
    n = len(arr)
    large = pa.types.is_large_list(arr.type)
    ow = 8 if large else 4
    off, pv, cv, _ = arrow_parts(arr)
    ent, masks, cmasks, cword, nulls = rev_list_reference(off, pv, cv)
    bufs = arr.buffers()
    child = arr.values
    cbufs = child.buffers()
    got = _run_list(bytes(bufs[1])[arr.offset * ow:(arr.offset + n + 1) * ow], large, n,
                    bytes(bufs[0]) if arr.null_count else None, arr.offset,
                    bytes(cbufs[0]) if child.null_count else None, child.offset + int(off[0]), cword)
    g_ent, g_masks, g_cmasks, g_nc, g_err = got
    assert g_err == 0
    assert np.array_equal(g_ent[:n], ent[:n])
    assert np.array_equal(g_masks, masks)
    assert np.array_equal(g_cmasks[: cmasks.shape[0]], cmasks)
    assert g_nc == nulls


@pytest.mark.parametrize("n,large,bit_off,child_off", [
    (1, False, 1, 0), (7, True, 5, 3), (2048, False, 64, 1), (2049, True, 2047, 7), (100_003, False, 5, 13), (100_003, True, 1, 0),
    (2049, False, 0, 0)])
def test_l0_rev_list_matches_the_restatement(n, large, bit_off, child_off):
    arr = make_list_array(n + bit_off + 3, 7 * n + bit_off, large, child_off).slice(bit_off, n)
    _check_l0(arr)


def test_l0_one_row_with_a_million_elements():
    lens = np.asarray([3, 1_200_001, 0, 5] + [2] * 3000)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    rng = np.random.default_rng(5)
    child = pa.array(rng.integers(0, 100, int(off[-1]), dtype=np.int32), mask=rng.random(int(off[-1])) < 0.1)
    arr = pa.ListArray.from_arrays(pa.array(off), child, mask=pa.array(rng.random(lens.shape[0]) < 0.2))
    _check_l0(arr.slice(1))


def test_l0_all_empty_lists():
    arr = pa.ListArray.from_arrays(pa.array(np.full(5001, 17, np.int32)), pa.array(np.arange(20, dtype=np.int32)))
    _check_l0(arr)


def test_l0_decreasing_offsets_raise_the_flag():
    off = np.arange(0, 3 * 5000, 3, dtype=np.int32)[:5000]
    off[3000] = off[2999] - 1
    cword = np.zeros(4, np.int64)
    for k in range(3):
        e0, e1 = off[k * 2048] - off[0], off[min((k + 1) * 2048, 4999)] - off[0]
        cword[k + 1] = cword[k] + (e1 - e0 + 63) // 64
    *_, err = _run_list(off.tobytes(), False, 4999, None, 0, None, 0, cword)
    assert err == 1


# ------------------------------------------------------------------------------------------- L1
def _plain(v, typ):
    """a pyarrow Python value in the form CollectedChunks.list_values decodes"""
    if v is None:
        return None
    if pa.types.is_decimal(typ):
        return int(v.scaleb(typ.scale))
    if pa.types.is_date32(typ):
        return (v - __import__("datetime").date(1970, 1, 1)).days
    return v


def _expected(arr):
    typ = arr.type.value_type
    if pa.types.is_timestamp(typ):
        arr = arr.cast(pa.list_(pa.int64()) if pa.types.is_list(arr.type) else pa.large_list(pa.int64()))
    return [None if row is None else [_plain(v, typ) for v in row] for row in arr.to_pylist()]


def _append(ctx, rb, type_ids, lists, dec_widths=None):
    """append `rb` (kept alive by the caller) and return the sink; `lists`: {col: (child_type, dec_width, dec_scale)}"""
    from duckdb_mbt_b200 import appender as ap
    sink = ap.CollectedChunks(type_ids, dec_widths, {c: (t, w) for c, (t, w, _) in lists.items()})
    a = ap.Appender(ctx, type_ids, sink)
    for c, (t, w, s) in lists.items():
        a.set_list(c, t, w, s)
    a.append_arrow(rb)
    a.flush()
    assert a.state == ap.FLUSHED and sink.nrows == len(rb)
    a.close()
    for c in lists:  # every entry stays inside its chunk's child vector
        for k, cnt in enumerate(sink.counts):
            e = np.frombuffer(sink.data[c][k], dtype=np.uint64).reshape(-1, 2)
            size = len(sink.child_data[c][k]) // ap._out_width(lists[c][0], lists[c][1])
            assert np.all(e[:cnt, 0] + e[:cnt, 1] <= size)
    return sink


def _child_values(type_name, m, rng):
    """(pyarrow child array of m values with NULLs, DuckDB child type, dec width, dec scale)"""
    nulls = rng.random(m) < 0.15
    pick = lambda f: [None if nulls[i] else f(i) for i in range(m)]  # noqa: E731
    if type_name == "INTEGER":
        return pa.array(rng.integers(-2**31, 2**31, m, dtype=np.int64).astype(np.int32), mask=nulls), ch.T_INTEGER, 0, 0
    if type_name == "BIGINT":
        return pa.array(rng.integers(-2**63, 2**63 - 1, m, dtype=np.int64), mask=nulls), ch.T_BIGINT, 0, 0
    if type_name == "BOOLEAN":
        return pa.array(rng.random(m) < 0.5, mask=nulls), ch.T_BOOLEAN, 0, 0
    if type_name == "DOUBLE":
        return pa.array(rng.standard_normal(m), mask=nulls), ch.T_DOUBLE, 0, 0
    if type_name == "DATE":
        return pa.array(rng.integers(-10**5, 10**5, m).astype(np.int32), mask=nulls).cast(pa.date32()), ch.T_DATE, 0, 0
    if type_name == "TIMESTAMP":
        return pa.array(rng.integers(0, 2 * 10**15, m, dtype=np.int64), mask=nulls).cast(pa.timestamp("us")), ch.T_TIMESTAMP, 0, 0
    if type_name.startswith("DECIMAL"):
        p, s = {"DECIMAL(9,2)": (9, 2), "DECIMAL(18,3)": (18, 3), "DECIMAL(38,0)": (38, 0)}[type_name]
        lim = 10**min(p, 30) - 1
        vals = pick(lambda i: decimal.Decimal(int(rng.integers(-2**62, 2**62)) % lim * (1 if i % 2 else -1)).scaleb(-s))
        return pa.array(vals, type=pa.decimal128(p, s)), ch.T_DECIMAL, p, s
    if type_name == "HUGEINT":
        return pa.array(pick(lambda i: decimal.Decimal(int(rng.integers(-2**62, 2**62)) * 10**16)), type=pa.decimal128(38, 0)), ch.T_HUGEINT, 0, 0
    if type_name == "VARCHAR":
        return pa.array(pick(lambda i: "x" * int(rng.integers(0, 30)) + str(i)), type=pa.string()), ch.T_VARCHAR, 0, 0
    if type_name == "BLOB":
        return pa.array(pick(lambda i: bytes(rng.integers(0, 256, int(rng.integers(0, 30)), dtype=np.uint8))), type=pa.binary()), ch.T_BLOB, 0, 0
    raise KeyError(type_name)


def _list_column(type_name, n, rng, large=False, max_len=6, child_off=3):
    lens = rng.integers(0, max_len + 1, n)
    off = np.concatenate([[0], np.cumsum(lens)])
    child, t, w, s = _child_values(type_name, int(off[-1]) + child_off, rng)
    typ = pa.LargeListArray if large else pa.ListArray
    arr = typ.from_arrays(pa.array(off, pa.int64() if large else pa.int32()), child.slice(child_off), mask=pa.array(rng.random(n) < 0.2))
    return arr, (t, w, s)


@pytest.mark.parametrize("type_name", ["INTEGER", "BIGINT", "BOOLEAN", "DOUBLE", "DATE", "TIMESTAMP", "DECIMAL(9,2)", "DECIMAL(18,3)",
                                       "DECIMAL(38,0)", "HUGEINT", "VARCHAR", "BLOB"])
def test_append_list_child_types_beside_scalar_columns(ctx, type_name):
    from test_gpu_appender import _oracle_column
    rng = np.random.default_rng(len(type_name))
    n = 9000
    lst, decl = _list_column(type_name, n, rng, large=type_name in ("BIGINT", "VARCHAR"))
    ids = pa.array(np.arange(n, dtype=np.int32), mask=rng.random(n) < 0.1)
    s = pa.array([None if i % 9 == 0 else "row %d of a batch" % i for i in range(n)])
    rb = pa.record_batch([ids, lst, s], names=["id", "l", "s"]).slice(11, n - 20)
    struct = rb.to_struct_array()
    sink = _append(ctx, struct, [ch.T_INTEGER, ch.T_LIST, ch.T_VARCHAR], {1: decl})
    assert sink.list_values(1) == _expected(struct.field(1))
    for c, t in ((0, ch.T_INTEGER), (2, ch.T_VARCHAR)):
        (exp_out, exp_val, _), w = _oracle_column(struct.field(c), t)
        assert sink.column_bytes(c) == exp_out.tobytes()[: rb.num_rows * w]
        assert np.array_equal(np.concatenate(sink.validity[c]), exp_val[: 32 * len(sink.counts)])


@pytest.mark.parametrize("env", [{"DMB_REV_BATCH_ROWS": "4096"}, {"DMB_REV_LIST_CHILD_CAP": "3000"},
                                 {"DMB_REV_BATCH_ROWS": "8192", "DMB_REV_LIST_CHILD_CAP": "20000"}])
def test_append_list_in_several_sub_batches(ctx, monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    rng = np.random.default_rng(77)
    n = 50_000
    a, da = _list_column("INTEGER", n, rng, max_len=4)
    b, db = _list_column("VARCHAR", n, rng, large=True, max_len=3)
    big = pa.ListArray.from_arrays(pa.array([0, 2, 40_002, 40_010], pa.int32()), pa.array(np.arange(40_010, dtype=np.int32)))
    a = pa.concat_arrays([a.slice(0, 30_000), big, a.slice(30_000)])  # one chunk far above the cap
    b = pa.concat_arrays([b.slice(0, 30_000), pa.array([["p"], None, ["q", None]], pa.large_list(pa.string())), b.slice(30_000)])
    rb = pa.record_batch([a, b], names=["a", "b"]).slice(3, n - 7)
    struct = rb.to_struct_array()
    sink = _append(ctx, struct, [ch.T_LIST, ch.T_LIST], {0: da, 1: db})
    assert sink.list_values(0) == _expected(struct.field(0))
    assert sink.list_values(1) == _expected(struct.field(1))


@pytest.mark.parametrize("layout", ["contiguous", "shuffled", "shared"])
def test_forward_then_reverse_round_trip_of_lists(ctx, layout):
    import list_cases
    from duckdb_mbt_b200 import arrow_result as ar
    lc = list_cases.make_list_column(12_345, 4, "ragged", 31, layout)
    batch = ch.ChunkBatch(lc.counts, [list_cases.as_column(lc, "l", ch.T_INTEGER)])
    res = ar.ArrowResult.from_chunks(ctx, batch)
    rb = res.to_record_batch()
    sink = _append(ctx, rb.to_struct_array(), [ch.T_LIST], {0: (ch.T_INTEGER, 0, 0)})
    res.close()
    expected = [None if row is None else [None if v is None else int.from_bytes(v, "little", signed=True) for v in row] for row in lc.expected]
    assert sink.list_values(0) == expected


# ------------------------------------------------------------------------------------------- refusals
def _failing_append(ctx, type_ids, rb, decl=None, sink=None):
    from duckdb_mbt_b200 import appender as ap
    from duckdb_mbt_b200.arrow_result import DuckDBError
    a = ap.Appender(ctx, type_ids, sink or ap.CollectedChunks(type_ids))
    if decl is not None:
        a.set_list(0, *decl)
    with pytest.raises(DuckDBError) as e:
        a.append_arrow(rb)
    assert a.state == ap.ERROR
    a.close()
    return str(e.value)


def test_refusals(ctx):
    from duckdb_mbt_b200 import appender as ap
    from duckdb_mbt_b200.arrow_result import DuckDBError
    ints = pa.record_batch([pa.array([[1, 2], None, []], pa.list_(pa.int32()))], names=["l"])
    assert "not declared" in _failing_append(ctx, [ch.T_LIST], ints)
    assert "does not match the declared child type" in _failing_append(ctx, [ch.T_LIST], ints, (ch.T_BIGINT, 0, 0))
    nested = pa.record_batch([pa.array([[[1], [2, 3]], None], pa.list_(pa.list_(pa.int32())))], names=["l"])
    assert "LIST<LIST>" in _failing_append(ctx, [ch.T_LIST], nested, (ch.T_INTEGER, 0, 0))
    structs = pa.record_batch([pa.array([[{"x": 1}], []], pa.list_(pa.struct([("x", pa.int32())])))], names=["l"])
    assert "LIST<STRUCT>" in _failing_append(ctx, [ch.T_LIST], structs, (ch.T_INTEGER, 0, 0))
    a = ap.Appender(ctx, [ch.T_LIST], ap.CollectedChunks([ch.T_LIST]))
    for t, name in ((ch.T_LIST, "LIST<LIST>"), (ch.T_STRUCT, "LIST<STRUCT>"), (ch.T_MAP, "LIST<MAP>")):
        with pytest.raises(DuckDBError, match=name):
            a.set_list(0, t)
    with pytest.raises(DuckDBError, match="only appendable through Arrow batches"):
        a.begin_row()
    a.close()


def test_decreasing_offsets_stop_before_the_sub_batch_reaches_the_sink(ctx, monkeypatch):
    from duckdb_mbt_b200 import appender as ap
    monkeypatch.setenv("DMB_REV_BATCH_ROWS", "4096")
    n = 20_000
    off = np.arange(0, 2 * (n + 1), 2, dtype=np.int32)
    off[10_300] = off[10_299] - 1  # inside chunk 5, i.e. sub-batch 2 (rows 8192..12287); chunk boundaries stay monotonic
    child = pa.array(np.arange(int(off[-1]), dtype=np.int32))
    arr = pa.Array.from_buffers(pa.list_(pa.int32()), n, [None, pa.py_buffer(off.tobytes())], children=[child])
    rb = pa.record_batch([arr], names=["l"])
    sink = ap.CollectedChunks([ch.T_LIST], None, {0: (ch.T_INTEGER, 0)})
    msg = _failing_append(ctx, [ch.T_LIST], rb, (ch.T_INTEGER, 0, 0), sink)
    assert "decrease" in msg
    assert sink.nrows == 8192  # sub-batches 0 and 1 only


# ------------------------------------------------------------------------------------------- glue + mock DuckDB
def test_glue_appends_list_columns_into_duckdb_vectors():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from test_glue_mock import Glue
    from duckdb_mbt_b200 import appender as ap
    g = Glue()
    vp = C.c_void_p
    g.mock.duckdb_mock_set_append_list_child.argtypes = [C.c_char_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32]
    g.mock.duckdb_mock_appended_list_child.restype = C.c_int64
    g.mock.duckdb_mock_appended_list_child.argtypes = [C.c_char_p, C.c_int64, C.c_int32, C.POINTER(vp), C.POINTER(vp)]
    types = np.asarray([ch.T_INTEGER, ch.T_LIST, ch.T_LIST], dtype=np.int32)
    assert g.mock.duckdb_mock_register_append_table(b"main", b"t_lists", 3, types.ctypes.data, None, None)
    assert g.mock.duckdb_mock_set_append_list_child(b"t_lists", 1, ch.T_INTEGER, 0, 0)
    assert g.mock.duckdb_mock_set_append_list_child(b"t_lists", 2, ch.T_VARCHAR, 0, 0)
    h = g.glue.duckdb_mb_appender_create(C.byref(g.conn), g.bytes_(b"main"), g.bytes_(b"t_lists"))
    assert h
    L = nat.lib()
    rng = np.random.default_rng(12)
    n = 5000
    li, _ = _list_column("INTEGER", n, rng)
    ls, _ = _list_column("VARCHAR", n, rng)
    struct = pa.record_batch([pa.array(np.arange(n, dtype=np.int32)), li, ls], names=["i", "li", "ls"]).slice(5, n - 9).to_struct_array()
    arr, sch = nat.ArrowArray(), nat.ArrowSchema()
    struct._export_to_c(C.addressof(arr), C.addressof(sch))
    try:
        ok = L.duckdb_mb_gpu_append_arrow_batch(vp(h), C.addressof(arr), C.addressof(sch))
    finally:
        ap._release(arr)
        ap._release(sch)
    assert ok, nat.moonbit_bytes(L.duckdb_mb_gpu_appender_error(vp(h)))
    assert L.duckdb_mb_gpu_appender_flush(vp(h))
    nrows = len(struct)
    nch = (nrows + 2047) // 2048
    assert g.mock.duckdb_mock_appended_rows(b"t_lists") == nrows and g.mock.duckdb_mock_appended_chunks(b"t_lists") == nch
    got = {1: [], 2: []}
    for k in range(nch):
        for c in (1, 2):
            dptr, mptr, cd, cm = vp(), vp(), vp(), vp()
            cnt = g.mock.duckdb_mock_appended_chunk(b"t_lists", k, c, C.byref(dptr), C.byref(mptr))
            size = g.mock.duckdb_mock_appended_list_child(b"t_lists", k, c, C.byref(cd), C.byref(cm))
            ent = np.frombuffer(C.string_at(dptr.value, cnt * 16), dtype=np.uint64).reshape(-1, 2)
            valid = np.unpackbits(np.frombuffer(C.string_at(mptr.value, 256), dtype=np.uint8), bitorder="little")[:cnt].astype(bool)
            nw = (size + 63) // 64
            cvalid = (np.unpackbits(np.frombuffer(C.string_at(cm.value, 8 * nw), dtype=np.uint8), bitorder="little")[:size].astype(bool)
                      if cm.value and nw else np.ones(size, bool))
            if c == 1:
                vals = np.frombuffer(C.string_at(cd.value, 4 * size), dtype=np.int32).tolist() if size else []
            else:
                raw = np.frombuffer(C.string_at(cd.value, 16 * size), dtype=np.uint8).reshape(-1, 16) if size else np.zeros((0, 16), np.uint8)
                vals = []
                for i in range(size):
                    ln = int(raw[i, 0:4].view(np.uint32)[0])
                    vals.append((bytes(raw[i, 4:4 + ln]) if ln <= 12 else C.string_at(int(raw[i, 8:16].view(np.uint64)[0]), ln)).decode()
                                if cvalid[i] else None)
            for r in range(cnt):
                o, ln = int(ent[r, 0]), int(ent[r, 1])
                assert o + ln <= size
                got[c].append([vals[j] if cvalid[j] else None for j in range(o, o + ln)] if valid[r] else None)
    assert got[1] == struct.field(1).to_pylist()
    assert got[2] == struct.field(2).to_pylist()
    L.duckdb_mb_begin_row.argtypes = [vp]
    assert L.duckdb_mb_begin_row(vp(h)) == 0
    assert b"only appendable through Arrow batches" in nat.moonbit_bytes(L.duckdb_mb_gpu_appender_error(vp(h)))
    L.duckdb_mb_appender_destroy.argtypes = [vp]
    L.duckdb_mb_appender_destroy(vp(h))
