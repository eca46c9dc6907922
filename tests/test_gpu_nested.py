"""Nested types through the host API (SURVEY.md 8f item 3; round-1 verdict item 8): STRUCT, LIST<VARCHAR>,
MAP = LIST<STRUCT<key, value>>, LIST<STRUCT>, LIST<LIST<x>>.  The reference rejects them on its chunk path
(src/duckdb_native.c:271-303) and has no Arrow mapping, so the contract is the Arrow format: every exported array is
validated in full by pyarrow and must read back as exactly the Python values the DuckDB-shaped vectors stand for."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
pa = pytest.importorskip("pyarrow")

from duckdb_mbt_b200 import chunks as ch  # noqa: E402

import list_cases  # noqa: E402
import nested_cases  # noqa: E402


@pytest.fixture(scope="module")
def ctx():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from duckdb_mbt_b200 import arrow_result as ar
    c = ar.GpuContext(0)
    yield c
    c.close()


def _export(ctx, counts, cols):
    from duckdb_mbt_b200 import arrow_result as ar
    batch = ch.ChunkBatch(counts, cols)
    with ar.ArrowResult.from_chunks(ctx, batch) as res:
        arrays = res.to_arrow()
    for a in arrays:
        a.validate(full=True)
    return arrays


@pytest.mark.parametrize("kind,arrow_type", [
    ("varchar", pa.list_(pa.string())),
    ("map", pa.map_(pa.string(), pa.int32())),
    ("struct", pa.list_(pa.struct([("a", pa.int32()), ("s", pa.string())]))),
    ("list", pa.list_(pa.list_(pa.int32()))),
    ("list_varchar", pa.list_(pa.list_(pa.string()))),
])
@pytest.mark.parametrize("n,pattern,layout", [(1, "full", "contiguous"), (2049, "full", "contiguous"), (9000, "ragged", "shuffled"),
                                              (40_001, "ragged", "contiguous")])
def test_list_children_that_are_not_one_fixed_vector(ctx, kind, arrow_type, n, pattern, layout):
    counts, col, expected = nested_cases.make_list_of(kind, n, pattern, 300 + n, layout)
    other = ch.fixed_column("i", ch.T_INTEGER, np.arange(n, dtype=np.int32), counts)
    arr, i = _export(ctx, counts, [col, other])
    assert arr.type.equals(arrow_type, check_metadata=False) or str(arr.type).replace("not null", "").replace(" ", "") == str(arrow_type).replace(" ", ""), arr.type
    assert len(arr) == n and arr.null_count == sum(1 for e in expected if e is None)
    assert arr.to_pylist() == expected
    assert i.to_pylist() == list(range(n))


@pytest.mark.parametrize("n,pattern", [(1, "full"), (5000, "ragged"), (30_011, "full")])
def test_struct_columns(ctx, n, pattern):
    counts, col, expected = nested_cases.make_struct(n, pattern, 40 + n)
    (arr,) = _export(ctx, counts, [col])
    assert pa.types.is_struct(arr.type) and [f.name for f in arr.type] == ["i", "s", "d", "inner"]
    assert arr.type.field("d").type == pa.decimal128(9, 2) and pa.types.is_struct(arr.type.field("inner").type)
    assert arr.null_count == sum(1 for e in expected if e is None)
    assert arr.to_pylist() == expected


def test_nested_columns_in_a_sharded_stream(ctx):
    """the slices of a nested column (shards / stream batches) carry their child levels with them"""
    from duckdb_mbt_b200 import arrow_result as ar
    n = 20_000
    counts, col, expected = nested_cases.make_list_of("map", n, "full", 77)
    counts2, st, exp_st = nested_cases.make_struct(n, "full", 78)
    batch = ch.ChunkBatch(counts, [col, st])
    with ar.ArrowResult.from_chunks(ctx, batch) as res:
        reader = res.to_stream(max_batch_rows=6000)
        got_m, got_s = [], []
        for b in reader:
            b.validate(full=True)
            got_m += b.column(0).to_pylist()
            got_s += b.column(1).to_pylist()
    assert got_m == expected and got_s == exp_st


def test_malformed_nested_entries_are_refused(ctx):
    from duckdb_mbt_b200 import arrow_result as ar
    counts, col, expected = nested_cases.make_list_of("varchar", 3000, "full", 5, null_frac=0.0)
    ent = col.data.view(np.uint64).reshape(-1, 2)
    ent[7] = (int(col.list_child_sizes[0]) - 1, 9)
    with ar.ArrowResult.from_chunks(ctx, ch.ChunkBatch(counts, [col])) as res:
        with pytest.raises(ar.DuckDBError, match="outside its chunk's child vector"):
            res.to_arrow(0)


def _int_rows(lc):
    return [None if row is None else [None if v is None else int.from_bytes(v, "little", signed=True) for v in row] for row in lc.expected]


@pytest.mark.parametrize("n,pattern,layout", [(9000, "ragged", "contiguous"), (6001, "full", "shuffled")])
def test_flat_and_described_list_of_integer_export_the_same_array(ctx, n, pattern, layout):
    """dmb_host_list's two forms of a fixed-width child (the flat child_* fields, child_col) are one column to the exporter"""
    lc = list_cases.make_list_column(n, 4, pattern, 600 + n, layout)
    other = ch.fixed_column("i", ch.T_INTEGER, np.arange(n, dtype=np.int32), lc.counts)
    flat, described, i = _export(ctx, lc.counts, [list_cases.as_column(lc, "l", ch.T_INTEGER),
                                                  list_cases.as_described_column(lc, "l", ch.T_INTEGER), other])
    assert flat.type == described.type == pa.list_(pa.field("item", pa.int32()))
    assert flat.equals(described)
    assert flat.to_pylist() == described.to_pylist() == _int_rows(lc)
    assert i.to_pylist() == list(range(n))


@pytest.mark.parametrize("child_type,dec_width,dec_scale", [(ch.T_INTEGER, 0, 0), (ch.T_DECIMAL, 9, 2)], ids=["integer", "decimal"])
def test_flat_list_in_stream_batches_across_chunks(ctx, child_type, dec_width, dec_scale):
    """record batches of a flat LIST column (every batch a slice of several ragged chunks) concatenate to the single export"""
    from duckdb_mbt_b200 import arrow_result as ar
    n = 20_000
    lc = list_cases.make_list_column(n, 4, "ragged", 71, "shuffled")
    batch = ch.ChunkBatch(lc.counts, [list_cases.as_column(lc, "l", child_type, dec_width, dec_scale)])
    with ar.ArrowResult.from_chunks(ctx, batch) as res:
        whole = res.to_arrow(0)
    with ar.ArrowResult.from_chunks(ctx, batch) as res:
        parts = []
        for b in res.to_stream(max_batch_rows=5000):
            b.validate()
            assert b.num_rows <= 5000
            parts.append(b.column(0))
    assert len(parts) > 2
    got = pa.concat_arrays(parts)
    assert got.type == whole.type
    assert got.to_pylist() == whole.to_pylist()
    if child_type == ch.T_INTEGER:
        assert got.to_pylist() == _int_rows(lc)


@pytest.mark.parametrize("stored_type,child_type", [(ch.T_UINTEGER, ch.T_ENUM), (ch.T_UUID, ch.T_LIST)], ids=["enum", "list"])
def test_flat_list_child_without_arrow_mapping_fails_at_export(ctx, stored_type, child_type):
    """a flat child whose type has no Arrow mapping here (ENUM, LIST given by type id) is accepted by from_chunks: the
    result still serves its other columns, and only the Arrow export of that column fails"""
    import ctypes as C
    from duckdb_mbt_b200 import arrow_result as ar
    from duckdb_mbt_b200 import native as nat
    n = 3000
    lc = list_cases.make_list_column(n, ch.PHYS_WIDTH[ch.phys_of_type(stored_type)], "ragged", 81, "contiguous")
    other = ch.fixed_column("i", ch.T_INTEGER, np.arange(n, dtype=np.int32), lc.counts)
    hb = ar.HostBatch(ch.ChunkBatch(lc.counts, [list_cases.as_column(lc, "l", stored_type), other]))
    hb._cols[0].list.contents.child_type_id = child_type  # (the Python batch builder only knows mapped child types)
    handle = ctx.lib.duckdb_mb_gpu_result_from_chunks(ctx.handle, C.byref(hb.struct))
    assert not ctx.lib.duckdb_mb_is_null_arrow_result(handle), nat.last_error()
    with ar.ArrowResult(ctx, handle, hb) as res:
        assert np.array_equal(res.get_column_int32(1), np.arange(n, dtype=np.int32))
        with pytest.raises(ar.DuckDBError, match="no Arrow mapping"):
            res.to_arrow(0)
        assert "LIST child type" in nat.last_error()
