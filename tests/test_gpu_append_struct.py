"""GPU: Arrow struct arrays appended to DuckDB STRUCT columns, checked against the restatement of
tests/test_rev_struct_cpu.py: rev_mask_kernel at L0, every accepted field type with NULL struct rows over non-zero field
payloads, struct / field / batch offsets, nesting three deep, ENUM fields and their errors, the forward -> reverse round
trip, the refusals, the glue on mock tables and one 20 M-row append."""
import ctypes as C
import itertools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
pa = pytest.importorskip("pyarrow")

import nested_cases  # noqa: E402
import reverse_semantics as rs  # noqa: E402
from duckdb_mbt_b200 import chunks as ch  # noqa: E402
from duckdb_mbt_b200 import native as nat  # noqa: E402
from test_rev_struct_cpu import NROWS, _nested, mask_and, struct_contract  # noqa: E402
from test_reverse_reference_cpu import APPEND_ROWS, PAIR_IDS, PAIRS, SUB_ROWS, column, placement  # noqa: E402

U8, U16 = ch.T_UTINYINT, ch.T_USMALLINT


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


def _spec(fs):
    name, t, *rest = fs
    return name, t, (rest[0] if rest else None)


def _declare(a, col, spec, decimals=None, path=()):
    """set_struct for `col` and every nested STRUCT; set_decimal / set_enum for DECIMAL (decimals: path -> (w, s)) and
    ENUM fields"""
    first = a.set_struct(col, [_spec(f)[1] for f in spec])
    for i, f in enumerate(spec):
        _, t, extra = _spec(f)
        if t == ch.T_STRUCT:
            _declare(a, first + i, extra, decimals, path + (i,))
        elif t == ch.T_DECIMAL and decimals and path + (i,) in decimals:
            a.set_decimal(first + i, *decimals[path + (i,)])
        elif t == ch.T_ENUM:
            a.set_enum(first + i, extra[1], extra[0])
    return first


def _append(ctx, batch, types, structs, decimals=None, enums=None):
    from duckdb_mbt_b200 import appender as ap
    sink = ap.CollectedChunks(types, structs=structs, enums=enums)
    a = ap.Appender(ctx, types, sink)
    for c, spec in structs.items():
        _declare(a, c, spec, (decimals or {}).get(c))
    for c, (it, labels) in (enums or {}).items():
        a.set_enum(c, labels, it)
    a.append_arrow(batch)
    a.flush()
    return sink, a


def _words(sink, key):
    return [bytes(m.tobytes()) for m in (sink.validity[key[0]] if len(key) == 1 else sink.field_validity[key])]


def _same(got, exp, what):
    if got == exp:
        return
    assert len(got) == len(exp), f"{what}: {len(got)} rows, expected {len(exp)}"
    i = next(i for i, (g, e) in enumerate(zip(got, exp)) if g != e)
    pytest.fail(f"{what}: row {i}: got {str(got[i])[:60]}, expected {str(exp[i])[:60]}")


def check_struct(sink, c, st, spec, decimals=None, path=()):
    """the masks and field vectors the sink received for STRUCT column c against struct_contract(st)"""
    con = struct_contract(st)
    key = (c,) + path
    bits = sink.valid_bits(c) if not path else sink.field_valid_bits(key)
    assert np.array_equal(bits, con[()][0]), f"{key}: struct mask"
    for k, cnt in enumerate(sink.counts):  # bits past count are zero
        assert not np.unpackbits(np.frombuffer(_words(sink, key)[k], np.uint8), bitorder="little")[cnt:].any()
    for i, f in enumerate(spec):
        _, t, extra = _spec(f)
        p = (i,)
        if t == ch.T_STRUCT:
            sub = {q[1:]: v for q, v in con.items() if q[:1] == p}
            _check_sub(sink, key + p, sub, extra, decimals, path + p)
        else:
            _check_leaf(sink, key + p, con[p], t, extra, decimals, path + p)


def _check_sub(sink, key, con, spec, decimals, path):
    assert np.array_equal(sink.field_valid_bits(key), con[()][0]), f"{key}: struct mask"
    for i, f in enumerate(spec):
        _, t, extra = _spec(f)
        if t == ch.T_STRUCT:
            _check_sub(sink, key + (i,), {q[1:]: v for q, v in con.items() if q[:1] == (i,)}, extra, decimals, path + (i,))
        else:
            _check_leaf(sink, key + (i,), con[(i,)], t, extra, decimals, path + (i,))


def _check_leaf(sink, key, vc, t, extra, decimals, path):
    valid, arr = vc
    if t == ch.T_ENUM:
        return  # ENUM fields: test_enum_fields
    table = (decimals or {}).get(path)
    dw = table[0] if table else (extra or 0)
    exp = [v if ok else None for v, ok in zip(rs.expected_cells(arr, t, table), valid)]
    got = []
    for k, cnt in enumerate(sink.counts):
        got += rs.decode_vector(sink.field_data[key][k], bytes(sink.field_validity[key][k].tobytes()), cnt, t, dw)
    _same(got, exp, f"field {key}")


# ------------------------------------------------------------------------------------------- L0: rev_mask_kernel
def _run_mask_jobs(jobs_spec, nrows):
    """jobs_spec: [(a bytes|None, a_off, b bytes|None, b_off, out_off)] -> output words per job (plus the 4 guard words)"""
    dev = torch.device("cuda")
    keep, outs = [], []
    jobs = (nat.RevMaskJob * len(jobs_spec))()
    nwords = ((63 + nrows + 2047) // 2048) * 32
    for j, (a, ao, b, bo, oo) in enumerate(jobs_spec):
        ta = torch.tensor(list(a), dtype=torch.uint8, device=dev) if a is not None else None
        tb = torch.tensor(list(b), dtype=torch.uint8, device=dev) if b is not None else None
        out = torch.full((nwords + 4,), 0x5A5A5A5A5A5A5A5A, dtype=torch.int64, device=dev)  # garbage the kernel must overwrite
        keep += [ta, tb]
        outs.append(out)
        jobs[j].in_a = ta.data_ptr() if ta is not None else None
        jobs[j].a_bit_offset = ao
        jobs[j].in_b = tb.data_ptr() if tb is not None else None
        jobs[j].b_bit_offset = bo
        jobs[j].out = out.data_ptr()
        jobs[j].out_bit_offset = oo
    dj = torch.frombuffer(bytearray(bytes(jobs)), dtype=torch.uint8).to(dev)
    assert nat.lib().dmb_dev_rev_mask_batch(dj.data_ptr(), C.addressof(jobs), len(jobs_spec), nrows, None) == 0, nat.last_error()
    torch.cuda.synchronize()
    return [o.cpu().numpy().view(np.uint64) for o in outs]


@pytest.mark.parametrize("nrows", NROWS[1:])
def test_mask_kernel_matches_the_restatement(ctx, nrows):
    rng = np.random.default_rng(nrows)
    nbytes = (nrows + 64) // 8 + 16
    a = rng.integers(0, 256, nbytes, dtype=np.uint8).tobytes()  # random bits everywhere: garbage around every slice
    b = rng.integers(0, 256, nbytes, dtype=np.uint8).tobytes()
    spec = [(a, off, b, (off * 37) % 64, off % 8) for off in range(64)]
    spec += [(None, 0, b, 5, 0), (a, 9, None, 0, 3), (None, 0, None, 0, 0)]
    outs = _run_mask_jobs(spec, nrows)
    for (ja, ao, jb, bo, oo), out in zip(spec, outs):
        exp = mask_and(ja, ao, jb, bo, nrows, oo)
        assert np.array_equal(out[:len(exp)], exp), (ao, bo, oo)
        assert (out[len(exp):] == 0x5A5A5A5A5A5A5A5A).all(), "wrote past its words"


def test_mask_kernel_refuses_bad_jobs(ctx):
    jobs = (nat.RevMaskJob * 1)()
    jobs[0].out_bit_offset = 64
    assert nat.lib().dmb_dev_rev_mask_batch(C.addressof(jobs), C.addressof(jobs), 1, 10, None) == -1
    assert "bit offset" in nat.last_error() or "no output" in nat.last_error()


# ------------------------------------------------------------------------------------------- every field type
def _struct_mask(n, shift):
    r = np.arange(n)
    null = ((r + shift) % 5 == 3) | np.isin(r, [0, 2047, 4095, 4096, n - 1][shift % 2::2])
    return null


def _pair_struct(typ, edges, j):
    """a batch of one STRUCT column of three fields of `typ` (field f at Arrow offset f + 1) under a NULL-struct pattern,
    the struct sliced by 2, and an INTEGER column"""
    e = len(edges)
    kids = []
    for f in range(3):
        idx, valid = placement(e, j, f)
        lead = f + 3
        full = column(typ, edges, np.concatenate([np.zeros(lead, np.int64), idx]), np.concatenate([np.ones(lead, bool), valid]))
        kids.append(full.slice(f + 1))
    n2 = APPEND_ROWS + 2
    st = pa.StructArray.from_arrays(kids, names=["f0", "f1", "f2"], mask=pa.array(np.concatenate([[False, False], _struct_mask(APPEND_ROWS, j)])))
    assert len(kids[0]) == n2
    st = st.slice(2)
    return pa.StructArray.from_arrays([st, pa.array(np.arange(APPEND_ROWS, dtype=np.int32))], names=["st", "i"])


@pytest.mark.parametrize("pair", PAIRS, ids=PAIR_IDS)
def test_every_field_type(ctx, monkeypatch, pair):
    monkeypatch.setenv("DMB_REV_BATCH_ROWS", str(SUB_ROWS))
    _, typ, type_id, table, edges = pair
    spec = [(f"f{f}", type_id, table[0]) if table else (f"f{f}", type_id) for f in range(3)]
    decimals = {0: {(f,): table for f in range(3)}} if table else None
    for j in range(2):  # the NULL-struct rows of one append are valid in the other
        batch = _pair_struct(typ, edges, j)
        sink, a = _append(ctx, batch, [ch.T_STRUCT, ch.T_INTEGER], {0: spec}, decimals)
        assert sink.counts == [2048, 2048, 2048, 1]
        assert sink.data[0] == [b""] * 4  # vec_data of a STRUCT column is NULL
        st = batch.field(0)
        con = struct_contract(st)
        fields_valid = [_valid_under(st, f) for f in range(3)]
        assert any((~con[()][0] & v).any() for v in fields_valid), "a NULL struct row over a valid field"
        check_struct(sink, 0, st, spec, decimals and decimals[0])
        assert np.array_equal(np.frombuffer(sink.column_bytes(1), np.int32), np.arange(APPEND_ROWS, dtype=np.int32))
        a.close()


def _valid_under(st, f):
    return np.asarray(st.field(f).is_valid().to_numpy(zero_copy_only=False), bool)


# ------------------------------------------------------------------------------------------- offsets
def test_batch_struct_and_field_offsets(ctx):
    rng = np.random.default_rng(3)
    n = 300
    spec = [("i", ch.T_INTEGER), ("b", ch.T_BOOLEAN), ("s", ch.T_VARCHAR)]
    for bo, so, fo in itertools.product(range(8), repeat=3):
        m = n + bo + so + 16
        i = pa.array(rng.integers(-99, 99, m).astype(np.int32), mask=rng.random(m) < 0.2).slice(fo)
        b = pa.array(rng.random(m) < 0.5, mask=rng.random(m) < 0.2).slice((fo + 3) % 8)
        s = pa.array([None if rng.random() < 0.2 else "x" * int(rng.integers(0, 20)) for _ in range(m)]).slice(7 - fo)
        k = m - 8
        st = pa.StructArray.from_arrays([i[:k], b[:k], s[:k]], names=["i", "b", "s"], mask=pa.array(rng.random(k) < 0.25)).slice(so)
        other = pa.array(np.arange(len(st), dtype=np.int32))
        batch = pa.StructArray.from_arrays([st, other], names=["st", "o"]).slice(bo, n)
        sink, a = _append(ctx, batch, [ch.T_STRUCT, ch.T_INTEGER], {0: spec})
        assert sink.nrows == n
        check_struct(sink, 0, batch.field(0), spec)
        a.close()


# ------------------------------------------------------------------------------------------- nesting
NESTED_SPEC = [("i", ch.T_INTEGER), ("b", ch.T_BOOLEAN), ("s", ch.T_VARCHAR),
               ("inner", ch.T_STRUCT, [("x", ch.T_BIGINT), ("inner2", ch.T_STRUCT, [("y", ch.T_BOOLEAN)])])]


@pytest.mark.parametrize("lead", [1, 2, 5, 8])
def test_three_levels_with_nulls_at_every_level(ctx, monkeypatch, lead):
    monkeypatch.setenv("DMB_REV_BATCH_ROWS", str(SUB_ROWS))
    rng = np.random.default_rng(100 + lead)
    st = _nested(rng, 10_000, lead)
    y = st.field(3).field(1).field(0)
    assert y.offset % 8 != 0 or lead == 8  # the BOOLEAN field's value bits start at another phase than bit 0
    sink, a = _append(ctx, pa.StructArray.from_arrays([st], names=["st"]), [ch.T_STRUCT], {0: NESTED_SPEC})
    check_struct(sink, 0, st, NESTED_SPEC)
    got = sink.struct_values(0)
    exp = st.to_pylist()
    con = struct_contract(st)
    for r in (0, 1, 2047, 2048, 4095, 4096, 9999):
        if con[()][0][r]:
            assert got[r]["i"] == exp[r]["i"] and got[r]["s"] == exp[r]["s"] and got[r]["b"] == exp[r]["b"]
        else:
            assert got[r] is None
    a.close()


def test_enum_fields(ctx, monkeypatch):
    from duckdb_mbt_b200.arrow_result import DuckDBError
    monkeypatch.setenv("DMB_REV_BATCH_ROWS", str(SUB_ROWS))
    labels = ["AIR", "MAIL", "SHIP"]
    n = 10_000
    idx = np.arange(n) % 3
    smask = np.arange(n) % 7 == 2
    spec = [("d", ch.T_ENUM, (U8, labels)), ("u", ch.T_ENUM, (U16, labels))]

    def batch(bad_row):
        di, ui = idx.copy(), [labels[k] for k in idx]
        di[bad_row] = 3  # outside the dictionary
        ui[bad_row + 1] = "RAIL"
        d = pa.DictionaryArray.from_arrays(pa.array(di.astype(np.int32)), pa.array(labels), safe=False)
        st = pa.StructArray.from_arrays([d, pa.array(ui)], names=["d", "u"], mask=pa.array(smask))
        return pa.StructArray.from_arrays([st], names=["st"])

    # under NULL struct rows: no error, the rows are NULL
    bad = 7 * 700 + 2
    smask[bad + 1] = True
    sink, a = _append(ctx, batch(bad), [ch.T_STRUCT], {0: spec})
    vals = sink.struct_values(0)
    assert [v is None for v in vals] == smask.tolist()
    assert all(v == {"d": labels[idx[r]], "u": labels[idx[r]]} for r, v in enumerate(vals) if v is not None)
    for f in range(2):
        pos = np.frombuffer(sink.field_bytes((0, f)), np.uint8 if f == 0 else np.uint16)
        assert not pos[smask].any() and not sink.field_valid_bits((0, f))[smask].any()
    a.close()
    # under a valid struct row: the append stops before that sub-batch, the message names the column, field path and row
    from duckdb_mbt_b200 import appender as ap
    for f, row, what in ((0, 5001, "index 3"), (1, 5003, "'RAIL'")):  # valid struct rows (row % 7 != 2)
        di, ui = idx.copy(), [labels[k] for k in idx]
        if f == 0:
            di[row] = 3
        else:
            ui[row] = "RAIL"
        assert not smask[row]
        st = pa.StructArray.from_arrays([pa.DictionaryArray.from_arrays(pa.array(di.astype(np.int32)), pa.array(labels), safe=False), pa.array(ui)],
                                        names=["d", "u"], mask=pa.array(smask))
        sink = ap.CollectedChunks([ch.T_STRUCT], structs={0: spec})
        a = ap.Appender(ctx, [ch.T_STRUCT], sink)
        _declare(a, 0, spec)
        with pytest.raises(DuckDBError) as e:
            a.append_arrow(pa.StructArray.from_arrays([st], names=["st"]))
        msg = str(e.value)
        assert f"column 0, field {f}, row {row}" in msg and what in msg and "column 1" not in msg and "column 2" not in msg, msg
        assert sink.nrows == 4096 and a.state == ap.ERROR
        a.close()


# ------------------------------------------------------------------------------------------- round trip
@pytest.mark.parametrize("n,pattern", [(1, "full"), (5000, "ragged"), (30_011, "full")])
def test_forward_export_then_append_round_trips(ctx, n, pattern):
    from duckdb_mbt_b200 import arrow_result as ar
    counts, col, expected = nested_cases.make_struct(n, pattern, 40 + n)
    with ar.ArrowResult.from_chunks(ctx, ch.ChunkBatch(counts, [col])) as res:
        (arr,) = res.to_arrow()
    spec = [("i", ch.T_INTEGER), ("s", ch.T_VARCHAR), ("d", ch.T_DECIMAL, 9), ("inner", ch.T_STRUCT, [("b", ch.T_BOOLEAN)])]
    decimals = {0: {(2,): (9, 2)}}
    sink, a = _append(ctx, pa.StructArray.from_arrays([arr], names=["st"]), [ch.T_STRUCT], {0: spec}, decimals)
    check_struct(sink, 0, arr, spec, decimals[0])
    assert arr.to_pylist() == expected
    got = sink.struct_values(0)
    want = [None if e is None else {"i": e["i"], "s": e["s"], "d": None if e["d"] is None else int(e["d"].scaleb(2)), "inner": e["inner"]}
            for e in expected]
    assert got == want
    a.close()


# ------------------------------------------------------------------------------------------- refusals
def test_refusals(ctx):
    from duckdb_mbt_b200 import appender as ap
    from duckdb_mbt_b200.arrow_result import DuckDBError
    two = pa.StructArray.from_arrays([pa.array([1, 2], pa.int32()), pa.array(["a", "b"])], names=["a", "b"])

    def appended(types, arrays, declare, match):
        a = ap.Appender(ctx, types, ap.CollectedChunks(types))
        declare(a)
        with pytest.raises(DuckDBError, match=match):
            a.append_arrow(pa.StructArray.from_arrays(arrays, names=[f"c{i}" for i in range(len(arrays))]))
        assert a.state == ap.ERROR
        a.close()

    appended([ch.T_STRUCT], [two], lambda a: None, r"column 0: the STRUCT column's fields are not declared \(duckdb_mb_gpu_appender_set_struct\)")
    appended([ch.T_STRUCT], [two], lambda a: a.set_struct(0, [ch.T_INTEGER]), "column 0: the Arrow struct has 2 fields, the STRUCT column 1")
    appended([ch.T_STRUCT], [two], lambda a: a.set_struct(0, [ch.T_INTEGER, ch.T_INTEGER]),
             "column 0, field 1: Arrow field format 'u' cannot be appended to a column of DuckDB type 4")
    nested = pa.StructArray.from_arrays([pa.array([1, 2], pa.int32()), pa.StructArray.from_arrays([pa.array([3, 4], pa.int32())], names=["z"])],
                                        names=["a", "n"])
    appended([ch.T_STRUCT], [nested], lambda a: a.set_struct(0, [ch.T_INTEGER, ch.T_STRUCT]),
             "column 0, field 1: the STRUCT column's fields are not declared")
    appended([ch.T_STRUCT], [two], lambda a: _declare(a, 0, [("a", ch.T_INTEGER), ("n", ch.T_STRUCT, [("z", ch.T_INTEGER)])]),
             "column 0, field 1: Arrow format 'u' cannot be appended to a STRUCT column")
    lst = pa.StructArray.from_arrays([pa.array([1, 2], pa.int32()), pa.array([[1], [2]])], names=["a", "l"])
    appended([ch.T_STRUCT], [lst], lambda a: a.set_struct(0, [ch.T_INTEGER, ch.T_VARCHAR]),
             r"column 0, field 1: an Arrow LIST field \('\+l'\) cannot be appended to a STRUCT")
    appended([ch.T_STRUCT], [pa.array([1, 2], pa.int32())], lambda a: a.set_struct(0, [ch.T_INTEGER]),
             "column 0: Arrow format 'i' cannot be appended to a STRUCT column")
    # a field shorter than the rows it is read at (pyarrow refuses to build one: shortened in the exported C struct)
    st = pa.StructArray.from_arrays([pa.StructArray.from_arrays([pa.array([1, 2, 3, 4], pa.int32())], names=["a"])], names=["c0"])
    a = ap.Appender(ctx, [ch.T_STRUCT], ap.CollectedChunks([ch.T_STRUCT]))
    a.set_struct(0, [ch.T_INTEGER])
    arr, sch = nat.ArrowArray(), nat.ArrowSchema()
    st._export_to_c(C.addressof(arr), C.addressof(sch))
    arr.children[0].contents.children[0].contents.length = 3
    try:
        with pytest.raises(DuckDBError, match=r"column 0, field 0 is shorter than the rows it is read at \(3 of 4\)"):
            a.append_arrow_c(C.addressof(arr), C.addressof(sch))
    finally:
        ap._release(arr)
        ap._release(sch)
    a.close()
    # declarations: refused by name, the handle stays usable
    a = ap.Appender(ctx, [ch.T_INTEGER, ch.T_STRUCT], ap.CollectedChunks([ch.T_INTEGER, ch.T_STRUCT]))
    for col, types, match in ((0, [ch.T_INTEGER], "column 0 is not a STRUCT column"), (1, [], "at least one field"),
                              (1, [ch.T_LIST], "LIST fields cannot be appended"), (1, [ch.T_INTEGER, 26], "field 1: MAP fields"),
                              (1, [ch.T_INTERVAL], "field type 15 cannot be appended"), (1, [28], "field type 28"),
                              (1, [33], "field type 33"), (5, [ch.T_INTEGER], "column 5 is not a STRUCT column")):
        with pytest.raises(DuckDBError, match=match):
            a.set_struct(col, types)
        assert a.state == ap.READY
    first = a.set_struct(1, [ch.T_INTEGER, ch.T_STRUCT])
    assert first == 2 and a.set_struct(1, [ch.T_INTEGER, ch.T_STRUCT]) == 2
    with pytest.raises(DuckDBError, match="column 1 already has a different STRUCT declaration"):
        a.set_struct(1, [ch.T_BIGINT, ch.T_STRUCT])
    assert a.set_struct(3, [ch.T_DECIMAL, ch.T_ENUM]) == 4  # a nested STRUCT: numbered after the fields so far
    a.set_decimal(4, 18, 3)
    a.set_enum(5, ["x"], U8)
    with pytest.raises(DuckDBError, match="is not a STRUCT column of a chunk being handed"):
        a.struct_field(1, 0)
    # the row protocol refuses the table
    with pytest.raises(DuckDBError, match="only appendable through Arrow batches"):
        a.begin_row()
    a.close()


# ------------------------------------------------------------------------------------------- glue + mock DuckDB
def _mock_read(g, table, k, col, path):
    vp = C.c_void_p
    d, m = vp(), vp()
    p = (C.c_int32 * len(path))(*path)
    cnt = g.mock.duckdb_mock_appended_struct_field(table, k, col, p, len(path), C.byref(d), C.byref(m))
    assert cnt >= 0
    return cnt, d.value, m.value


def test_glue_appends_struct_columns():
    from test_glue_mock import Glue
    from duckdb_mbt_b200 import appender as ap
    g = Glue()
    vp, i32p = C.c_void_p, C.POINTER(C.c_int32)
    g.mock.duckdb_mock_set_append_struct.argtypes = [C.c_char_p, C.c_int32, i32p, C.c_int32, C.c_int32, i32p, i32p, i32p]
    g.mock.duckdb_mock_set_append_enum_field.argtypes = [C.c_char_p, C.c_int32, i32p, C.c_int32, C.c_int32, C.c_uint32, vp]
    g.mock.duckdb_mock_appended_struct_field.restype = C.c_int64
    g.mock.duckdb_mock_appended_struct_field.argtypes = [C.c_char_p, C.c_int64, C.c_int32, i32p, C.c_int32, C.POINTER(vp), C.POINTER(vp)]
    ints = lambda xs: (C.c_int32 * len(xs))(*xs)  # noqa: E731
    table = b"t_struct"
    types = np.asarray([ch.T_INTEGER, ch.T_STRUCT, ch.T_STRUCT], dtype=np.int32)
    assert g.mock.duckdb_mock_register_append_table(b"main", table, 3, types.ctypes.data, None, None)
    assert g.mock.duckdb_mock_set_append_struct(table, 1, None, 0, 4, ints([ch.T_INTEGER, ch.T_VARCHAR, ch.T_DECIMAL, ch.T_ENUM]),
                                                ints([0, 0, 18, 0]), ints([0, 0, 3, 0]))
    labels = ["red", "green", "blue"]
    bufs = [C.create_string_buffer(x.encode()) for x in labels]
    ptrs = (C.c_char_p * 3)(*[C.cast(b, C.c_char_p) for b in bufs])
    assert g.mock.duckdb_mock_set_append_enum_field(table, 1, ints([3]), 1, 1, 3, C.cast(ptrs, vp))
    assert g.mock.duckdb_mock_set_append_struct(table, 2, None, 0, 2, ints([ch.T_BIGINT, ch.T_STRUCT]), None, None)
    assert g.mock.duckdb_mock_set_append_struct(table, 2, ints([1]), 1, 2, ints([ch.T_BOOLEAN, ch.T_VARCHAR]), None, None)
    h = g.glue.duckdb_mb_appender_create(C.byref(g.conn), g.bytes_(b"main"), g.bytes_(table))
    assert h
    rng = np.random.default_rng(9)
    n = 5000
    from decimal import Decimal
    s1 = pa.StructArray.from_arrays(
        [pa.array(rng.integers(-9, 9, n).astype(np.int32), mask=rng.random(n) < 0.1),
         pa.array([None if rng.random() < 0.1 else "long string number %d!" % k for k in range(n)]),
         pa.array([None if k % 9 == 0 else Decimal(k * 7 - 3000).scaleb(-3) for k in range(n)], pa.decimal128(18, 3)),
         pa.DictionaryArray.from_arrays(pa.array((np.arange(n) % 3).astype(np.int8), mask=np.arange(n) % 11 == 0), pa.array(labels))],
        names=["i", "s", "d", "e"], mask=pa.array(rng.random(n) < 0.2))
    inner = pa.StructArray.from_arrays([pa.array(rng.random(n + 3) < 0.5, mask=rng.random(n + 3) < 0.1).slice(3),
                                        pa.array(["inner text over twelve %d" % k if k % 4 else None for k in range(n)])],
                                       names=["b", "t"], mask=pa.array(rng.random(n) < 0.2))
    s2 = pa.StructArray.from_arrays([pa.array(np.arange(n, dtype=np.int64)), inner], names=["x", "inner"], mask=pa.array(rng.random(n) < 0.1))
    batch = pa.StructArray.from_arrays([pa.array(np.arange(n, dtype=np.int32)), s1, s2], names=["k", "s1", "s2"])
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

    def read(col, path, t, dw=0):
        out, valid = [], []
        for k in range(nch):
            if path:
                cnt, d, m = _mock_read(g, table, k, col, path)
            else:
                d, m = vp(), vp()
                cnt = g.mock.duckdb_mock_appended_chunk(table, k, col, C.byref(d), C.byref(m))
                d, m = d.value, m.value
            mask = C.string_at(m, 256) if m else None
            valid += [True] * cnt if mask is None else [bool(mask[i >> 3] >> (i & 7) & 1) for i in range(cnt)]
            if t is not None:
                w = rs.vector_width(t, dw)
                out += rs.decode_vector(C.string_at(d, cnt * w), mask, cnt, t, dw, strict=False)
        return out, valid

    for col, st, leaves in ((1, s1, {(0,): (ch.T_INTEGER, None), (1,): (ch.T_VARCHAR, None), (2,): (ch.T_DECIMAL, (18, 3))}),
                            (2, s2, {(0,): (ch.T_BIGINT, None), (1, 0): (ch.T_BOOLEAN, None), (1, 1): (ch.T_VARCHAR, None)})):
        con = struct_contract(st)
        assert read(col, (), None)[1] == con[()][0].tolist()
        for path, (t, table_dec) in leaves.items():
            valid, a = con[path]
            got, gvalid = read(col, path, t, table_dec[0] if table_dec else 0)
            assert gvalid == valid.tolist(), path
            assert got == [v if ok else None for v, ok in zip(rs.expected_cells(a, t, table_dec), valid)], path
    assert read(2, (1,), None)[1] == struct_contract(s2)[(1,)][0].tolist()
    # the ENUM field: positions, NULL under NULL structs and NULL indices
    pos, evalid = [], []
    for k in range(nch):
        cnt, d, m = _mock_read(g, table, k, 1, [3])
        pos += list(np.frombuffer(C.string_at(d, cnt), np.uint8))
        mask = C.string_at(m, 256)
        evalid += [bool(mask[i >> 3] >> (i & 7) & 1) for i in range(cnt)]
    svalid = struct_contract(s1)[()][0]
    want = svalid & (np.arange(n) % 11 != 0)
    assert evalid == want.tolist()
    assert [int(p) for p, ok in zip(pos, evalid) if ok] == [int(k % 3) for k, ok in zip(range(n), want) if ok]
    L.duckdb_mb_appender_destroy.argtypes = [vp]
    L.duckdb_mb_appender_destroy(vp(h))


# ------------------------------------------------------------------------------------------- scale
def test_twenty_million_rows(ctx):
    rng = np.random.default_rng(20)
    n = 20_000_000
    labels = ["AIR", "FOB", "MAIL", "RAIL", "REG AIR", "SHIP", "TRUCK"]
    smask = rng.random(n) < 0.1
    iv, dv, sv, ev = (rng.random(n) >= 0.05 for _ in range(4))
    i = rng.integers(-2**31, 2**31 - 1, n).astype(np.int32)
    d = rng.random(n)
    e = rng.integers(0, len(labels), n).astype(np.uint8)
    s = pa.DictionaryArray.from_arrays(pa.array(e, mask=~sv), pa.array(labels)).cast(pa.string())
    st = pa.StructArray.from_arrays([pa.array(i, mask=~iv), pa.array(d, mask=~dv), s,
                                     pa.DictionaryArray.from_arrays(pa.array(e, mask=~ev), pa.array(labels))],
                                    names=["i", "d", "s", "e"], mask=pa.array(smask))
    spec = [("i", ch.T_INTEGER), ("d", ch.T_DOUBLE), ("s", ch.T_VARCHAR), ("e", ch.T_ENUM, (U8, labels))]
    sink, a = _append(ctx, pa.StructArray.from_arrays([st], names=["st"]), [ch.T_STRUCT], {0: spec})
    ok = ~smask
    assert np.array_equal(sink.valid_bits(0), ok)
    assert np.array_equal(sink.field_valid_bits((0, 0)), ok & iv)
    assert np.array_equal(np.frombuffer(sink.field_bytes((0, 0)), np.int32), np.where(ok & iv, i, 0))
    assert np.array_equal(sink.field_valid_bits((0, 1)), ok & dv)
    assert np.array_equal(np.frombuffer(sink.field_bytes((0, 1)), np.float64), np.where(ok & dv, d, 0.0))
    assert np.array_equal(sink.field_valid_bits((0, 3)), ok & ev)
    assert np.array_equal(np.frombuffer(sink.field_bytes((0, 3)), np.uint8), np.where(ok & ev, e, 0))
    assert np.array_equal(sink.field_valid_bits((0, 2)), ok & sv)
    for r0 in (0, 4 << 20, n // 2 - 1000, n - 3000):  # sampled windows of the strings, across sub-batch boundaries
        k0, k1 = r0 // 2048, min((r0 + 3000 + 2047) // 2048, len(sink.counts))
        rows = []
        for k in range(k0, k1):
            rows += rs.decode_vector(sink.field_data[(0, 2)][k], bytes(sink.field_validity[(0, 2)][k].tobytes()), sink.counts[k], ch.T_VARCHAR)
        want = [labels[e[r]].encode() if ok[r] and sv[r] else None for r in range(k0 * 2048, k0 * 2048 + len(rows))]
        assert rows == want, r0
    a.close()
