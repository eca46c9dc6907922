"""GPU: the appender's Arrow -> DataChunk conversions (rev_fixed_kernel, rev_string_kernel, rev_list_kernel and the
host mapping in host_appender.cu) against tests/reverse_semantics.py, with the table's column types declared.

Every (Arrow type, column type) pair the appender accepts is appended with its edge set placed by
tests/test_reverse_reference_cpu.py: each edge value lands at row 0 and row 2047 of a chunk, at the first and last
row of a sub-batch (DMB_REV_BATCH_ROWS=4096), in rev_copy's scalar tail, in columns whose Arrow offsets differ, and
both valid and NULL over a non-zero payload.  The same edge sets go through LIST children, at each chunk's first child
element and across DMB_REV_LIST_CHILD_CAP cuts.  Then the decimal refusals by name, and the glue appending DECIMAL
columns of a mock table at the table's own width and scale."""
import ctypes as C
from decimal import Decimal

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
pa = pytest.importorskip("pyarrow")

import reverse_semantics as rs  # noqa: E402
from duckdb_mbt_b200 import chunks as ch  # noqa: E402
from duckdb_mbt_b200 import native as nat  # noqa: E402
from test_reverse_reference_cpu import (APPEND_ROWS, NCOLS, PAIR_IDS, PAIRS, SUB_ROWS, appends_for, column,  # noqa: E402
                                        decimal_values, stride_for, struct_for)


@pytest.fixture(scope="module")
def ctx():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from duckdb_mbt_b200 import arrow_result as ar
    c = ar.GpuContext(0)
    yield c
    c.close()


def _short(v):
    return v if not isinstance(v, (bytes, list)) or len(v) <= 24 else f"{type(v).__name__} of {len(v)}: {v[:16]!r}..."


def _same(got: list, exp: list, what: str) -> None:
    """list equality, reported at the first row that differs"""
    if got == exp:
        return
    if len(got) != len(exp):
        pytest.fail(f"{what}: {len(got)} rows, expected {len(exp)}")
    i = next(i for i, (g, e) in enumerate(zip(got, exp)) if g != e)
    pytest.fail(f"{what}: row {i} (row {i % APPEND_ROWS} of its append): got {_short(got[i])}, expected {_short(exp[i])}")


@pytest.mark.parametrize("pair", PAIRS, ids=PAIR_IDS)
def test_append_matches_the_reference(ctx, monkeypatch, pair):
    from duckdb_mbt_b200 import appender as ap
    monkeypatch.setenv("DMB_REV_BATCH_ROWS", str(SUB_ROWS))
    _, typ, type_id, table, edges = pair
    dw = table[0] if table else 0
    types = [type_id] * NCOLS
    for j in range(appends_for(len(edges))):  # one appender per append: a batch's strings are checked while it is alive
        sink = ap.CollectedChunks(types, [dw] * NCOLS)
        a = ap.Appender(ctx, types, sink)
        if table:
            for c in range(NCOLS):
                a.set_decimal(c, *table)
        struct = struct_for(typ, edges, j)
        a.append_arrow(struct)
        a.flush()
        assert sink.nrows == APPEND_ROWS and sink.counts == [2048, 2048, 2048, 1]
        for c in range(NCOLS):
            _same(rs.decode_collected(sink, c, type_id, dw), rs.expected_cells(struct.field(c), type_id, table), f"append {j} column {c}")
        a.close()


# ------------------------------------------------------------------------------------------- LIST children
LIST_CAP = 40  # DMB_REV_LIST_CHILD_CAP: below one chunk's 65 elements, so every chunk is a sub-batch of its own


def _list_of_edges(typ, edges: list, large: bool):
    """E + 1 chunks of lists; chunk m's child elements start with edge m % E and hold 65 elements (rows 0 (two), every
    64th row, and NULL rows at 32 mod 64 over a one-element Arrow segment); 65 % (16 / w) == 1 puts the last one in
    rev_copy's tail"""
    e = len(edges)
    s = stride_for(e)
    nch = e + 1
    n = nch * 2048
    i = np.arange(n) % 2048
    lens = np.where(i == 0, 2, np.where(i % 32 == 0, 1, 0))
    valid = i % 64 != 32
    idx, cvalid = [], []
    for m in range(nch):
        k = np.arange(65)
        idx.append((m + k * s) % e)
        cvalid.append(k % 7 != 3)
    idx, cvalid = np.concatenate(idx), np.concatenate(cvalid)
    lead = 3  # the child array starts at Arrow offset 3
    child = column(typ, edges, np.concatenate([np.zeros(lead, np.int64), idx]), np.concatenate([np.ones(lead, bool), cvalid])).slice(lead)
    off = np.concatenate([[0], np.cumsum(lens)])
    cls = pa.LargeListArray if large else pa.ListArray
    return cls.from_arrays(pa.array(off, pa.int64() if large else pa.int32()), child, mask=pa.array(~valid))


@pytest.mark.parametrize("pair", PAIRS, ids=PAIR_IDS)
def test_list_children_match_the_reference(ctx, monkeypatch, pair):
    from duckdb_mbt_b200 import appender as ap
    monkeypatch.setenv("DMB_REV_BATCH_ROWS", str(SUB_ROWS))
    monkeypatch.setenv("DMB_REV_LIST_CHILD_CAP", str(LIST_CAP))
    _, typ, type_id, table, edges = pair
    dw, ds = table if table else (0, 0)
    lst = _list_of_edges(typ, edges, large=len(edges) % 2 == 1)
    struct = pa.StructArray.from_arrays([lst], names=["l"])
    sink = ap.CollectedChunks([ch.T_LIST], None, {0: (type_id, dw)})
    a = ap.Appender(ctx, [ch.T_LIST], sink)
    a.set_list(0, type_id, dw, ds)
    a.append_arrow(struct)
    a.flush()
    assert sink.nrows == len(lst)
    _same(rs.decode_collected(sink, 0, ch.T_LIST, child=(type_id, dw)), rs.expected_lists(struct.field(0), type_id, table), "LIST")
    a.close()


# ------------------------------------------------------------------------------------------- refusals
# (id, Arrow type, column type, the table's DECIMAL (w, s) or None, its Arrow format, what the refusal names)
REFUSALS = [
    ("decimal32", pa.decimal32(9, 2), ch.T_DECIMAL, (9, 2), "d:9,2,32", "32-bit"),
    ("decimal64", pa.decimal64(18, 2), ch.T_DECIMAL, (18, 2), "d:18,2,64", "64-bit"),
    ("decimal256", pa.decimal256(40, 2), ch.T_DECIMAL, (38, 2), "d:40,2,256", "256-bit"),
    ("decimal256-hugeint", pa.decimal256(38, 0), ch.T_HUGEINT, None, "d:38,0,256", "256-bit"),
    ("scale", pa.decimal128(18, 3), ch.T_DECIMAL, (18, 2), "d:18,3", "scale 3"),
    ("smaller-scale", pa.decimal128(9, 1), ch.T_DECIMAL, (18, 2), "d:9,1", "scale 1"),
    ("precision", pa.decimal128(38, 2), ch.T_DECIMAL, (18, 2), "d:38,2", "precision 38"),
    ("precision-class", pa.decimal128(5, 2), ch.T_DECIMAL, (4, 2), "d:5,2", "precision 5"),
    ("hugeint-scale", pa.decimal128(20, 4), ch.T_HUGEINT, None, "d:20,4", "scale 4"),
]


def _refused(ctx, types, batch, declare) -> str:
    from duckdb_mbt_b200 import appender as ap
    from duckdb_mbt_b200.arrow_result import DuckDBError
    sink = ap.CollectedChunks([ch.T_INTEGER] * len(types))
    a = ap.Appender(ctx, types, sink)
    declare(a)
    with pytest.raises(DuckDBError) as e:
        a.append_arrow(batch)
    assert a.state == ap.ERROR and sink.nrows == 0
    a.close()
    return str(e.value)


@pytest.mark.parametrize("case", REFUSALS, ids=[r[0] for r in REFUSALS])
def test_decimal_refusals_name_the_column_and_the_format(ctx, case):
    _, typ, type_id, table, fmt, why = case
    vals = pa.array([Decimal(1).scaleb(-typ.scale), None], typ)
    ids = pa.array([1, 2], pa.int32())
    top = pa.record_batch([ids, vals], names=["i", "d"])
    msg = _refused(ctx, [ch.T_INTEGER, type_id], top, lambda a: table and a.set_decimal(1, *table))
    assert "column 1" in msg and f"'{fmt}'" in msg and why in msg, msg
    assert rs.decimal_refusal(typ.precision, typ.scale, typ.bit_width, type_id, table) is not None
    lst = pa.ListArray.from_arrays(pa.array([0, 1, 2], pa.int32()), vals)
    nested = pa.record_batch([ids, lst], names=["i", "l"])
    msg = _refused(ctx, [ch.T_INTEGER, ch.T_LIST], nested, lambda a: a.set_list(1, type_id, *(table or (0, 0))))
    assert "column 1" in msg and f"'{fmt}'" in msg and why in msg, msg


def test_an_undeclared_decimal_column_is_declared_by_its_first_batch(ctx):
    from duckdb_mbt_b200 import appender as ap
    from duckdb_mbt_b200.arrow_result import DuckDBError
    first = pa.array([Decimal("-9999.9"), Decimal("0.1"), None], pa.decimal128(5, 1))
    sink = ap.CollectedChunks([ch.T_DECIMAL], [5])
    a = ap.Appender(ctx, [ch.T_DECIMAL], sink)
    a.append_arrow(pa.record_batch([first], names=["d"]))
    a.append_arrow(pa.record_batch([pa.array([Decimal("12.3")], pa.decimal128(3, 1))], names=["d"]))  # narrower: fits DECIMAL(5,1)
    a.flush()
    assert rs.decode_collected(sink, 0, ch.T_DECIMAL, 5) == [-99999, 1, None, 123]  # int32 cells: DECIMAL(5,1)
    for later, why in ((pa.decimal128(5, 2), "scale 2"), (pa.decimal128(6, 1), "precision 6")):
        b = ap.Appender(ctx, [ch.T_DECIMAL], ap.CollectedChunks([ch.T_DECIMAL], [5]))
        b.append_arrow(pa.record_batch([first], names=["d"]))
        with pytest.raises(DuckDBError, match=why):
            b.append_arrow(pa.record_batch([pa.array([Decimal(1)], later)], names=["d"]))
        b.close()
    a.close()


# ------------------------------------------------------------------------------------------- glue + mock DuckDB
def test_glue_appends_decimals_at_the_table_width_and_scale():
    """A mock table declares DECIMAL(4,1), DECIMAL(9,2), DECIMAL(18,3), DECIMAL(38,10), HUGEINT and
    LIST<DECIMAL(18,3)>; the batches carry smaller precisions at the table's scales, as pyarrow infers them from Python
    Decimals.  What the table holds, read back at its own widths, is the reference's."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from test_glue_mock import Glue
    from duckdb_mbt_b200 import appender as ap
    g = Glue()
    vp = C.c_void_p
    g.mock.duckdb_mock_set_append_list_child.argtypes = [C.c_char_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32]
    g.mock.duckdb_mock_appended_list_child.restype = C.c_int64
    g.mock.duckdb_mock_appended_list_child.argtypes = [C.c_char_p, C.c_int64, C.c_int32, C.POINTER(vp), C.POINTER(vp)]
    decls = [(ch.T_DECIMAL, 4, 1, 2), (ch.T_DECIMAL, 9, 2, 4), (ch.T_DECIMAL, 18, 3, 5), (ch.T_DECIMAL, 38, 10, 12), (ch.T_HUGEINT, 38, 0, 20)]
    types = np.asarray([t for t, *_ in decls] + [ch.T_LIST], dtype=np.int32)
    widths = np.asarray([w if t == ch.T_DECIMAL else 0 for t, w, _, _ in decls] + [0], dtype=np.int32)
    scales = np.asarray([s for _, _, s, _ in decls] + [0], dtype=np.int32)
    assert g.mock.duckdb_mock_register_append_table(b"main", b"t_decimals", len(types), types.ctypes.data, widths.ctypes.data, scales.ctypes.data)
    assert g.mock.duckdb_mock_set_append_list_child(b"t_decimals", len(decls), ch.T_DECIMAL, 18, 3)
    h = g.glue.duckdb_mb_appender_create(C.byref(g.conn), g.bytes_(b"main"), g.bytes_(b"t_decimals"))
    assert h
    L = nat.lib()
    n = 5000
    r = np.arange(n)
    cols = []
    for t, w, s, p in decls:
        edges = decimal_values(p, s)
        vals = [None if i % 11 == 5 else edges[(i * stride_for(len(edges))) % len(edges)] for i in r]
        cols.append(pa.array(vals).cast(pa.decimal128(p, s)))
    child_edges = decimal_values(5, 3)
    child = pa.array([None if i % 9 == 4 else child_edges[i % len(child_edges)] for i in range(2 * n)]).cast(pa.decimal128(5, 3))
    cols.append(pa.ListArray.from_arrays(pa.array(2 * np.arange(n + 1), pa.int32()), child, mask=pa.array(r % 13 == 6)))
    struct = pa.record_batch(cols, names=[f"c{i}" for i in range(len(cols))]).slice(3, n - 7).to_struct_array()
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
    assert g.mock.duckdb_mock_appended_rows(b"t_decimals") == nrows
    for c, (t, w, s, _) in enumerate(decls):
        got = []
        for k in range(nch):
            dptr, mptr = vp(), vp()
            cnt = g.mock.duckdb_mock_appended_chunk(b"t_decimals", k, c, C.byref(dptr), C.byref(mptr))
            mask = C.string_at(mptr.value, 256) if mptr.value else None
            got += rs.decode_vector(C.string_at(dptr.value, 2048 * rs.vector_width(t, w)), mask, cnt, t, w, strict=False)
        _same(got, rs.expected_cells(struct.field(c), t, (w, s) if t == ch.T_DECIMAL else None), f"DuckDB column {c}")
    c = len(decls)
    got = []
    for k in range(nch):
        dptr, mptr, cd, cm = vp(), vp(), vp(), vp()
        cnt = g.mock.duckdb_mock_appended_chunk(b"t_decimals", k, c, C.byref(dptr), C.byref(mptr))
        size = g.mock.duckdb_mock_appended_list_child(b"t_decimals", k, c, C.byref(cd), C.byref(cm))
        cmask = C.string_at(cm.value, 8 * ((size + 63) // 64)) if cm.value and size else None
        got += rs.decode_list_vector(C.string_at(dptr.value, 16 * cnt), C.string_at(mptr.value, 256) if mptr.value else None, cnt,
                                     C.string_at(cd.value, 8 * size) if size else b"", cmask, size, ch.T_DECIMAL, 18, strict=False)
    _same(got, rs.expected_lists(struct.field(c), ch.T_DECIMAL, (18, 3)), "DuckDB LIST<DECIMAL(18,3)>")
    L.duckdb_mb_appender_destroy.argtypes = [vp]
    L.duckdb_mb_appender_destroy(vp(h))
