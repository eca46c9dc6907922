"""ENUM columns (SURVEY.md §8f item 3): uint8/16/32 index vectors + the type's dictionary.
The reference keeps an ENUM cell as Value::String of its label (src/duckdb_parsing.mbt:119-122), gets the label
through duckdb_value_varchar (src/duckdb_native.c:215-238, :2474-2510) and names the column "string" in the Arrow
schema JSON (:2314-2339).  Here: one lookup kernel (kernels_enum.cu) + the string kernels with the dictionary as
the heap; the Arrow C Data export is dictionary-encoded.  Checked against the oracle's restatement (UNPINNED in
the reference: no reference test holds an ENUM column) and with pyarrow."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
pa = pytest.importorskip("pyarrow")

import oracle  # noqa: E402
from duckdb_mbt_b200 import chunks as ch  # noqa: E402


@pytest.fixture(scope="module")
def ctx():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from duckdb_mbt_b200 import arrow_result as ar
    c = ar.GpuContext(0)
    yield c
    c.close()


def _result(ctx, batch, **kw):
    from duckdb_mbt_b200 import arrow_result as ar
    return ar.ArrowResult.from_chunks(ctx, batch, **kw)


def _labels(k, rng, max_len):
    out = []
    for i in range(k):
        ln = int(rng.integers(1, max_len + 1))
        body = rng.integers(0x61, 0x7B, max_len, dtype=np.uint8).tobytes()
        out.append((b"%d_" % i + body)[:ln])
    if k > 2:
        out[1] = b""  # an empty label is legal bytes-wise and exercises zero-length entries
    return out


def _enum_batch(n, k, max_len, pattern, seed, null_frac=0.2):
    rng = np.random.default_rng(seed)
    counts = ch.chunk_counts(n, pattern, rng)
    labels = _labels(k, rng, max_len)
    idx = rng.integers(0, k, n)
    valid = rng.random(n) >= null_frac if null_frac else None
    # garbage under NULL rows stays inside the index type but may point past the dictionary
    col = ch.enum_column("e", labels, idx, counts, valid=valid, garbage_rng=rng if valid is not None else None)
    other = ch.fixed_column("i", ch.T_INTEGER, np.arange(n, dtype=np.int32), counts)
    return ch.ChunkBatch(counts, [col, other]), labels, idx, valid


@pytest.mark.parametrize("n,k,max_len,pattern", [
    (1, 1, 3, "full"), (2049, 3, 8, "full"), (10_000, 7, 12, "ragged"),      # every label inlined: the heap-less kernel
    (40_001, 5, 30, "ragged"), (100_000, 300, 20, "full"),                      # uint16 indices, labels in the heap
    (30_000, 70_000, 9, "ragged"), (20_000, 4, 200, "full")])                   # uint32 indices; labels longer than a render slot
def test_enum_string_getter_and_text_column(ctx, n, k, max_len, pattern):
    from duckdb_mbt_b200 import typed_result as tr
    batch, labels, idx, valid = _enum_batch(n, k, max_len, pattern, 77 + n + k)
    assert batch.columns[0].phys == (ch.P_U8 if k <= 256 else ch.P_U16 if k <= 65536 else ch.P_U32)
    ora = oracle.OracleResult(batch)
    with _result(ctx, batch) as res:
        for nullable in (False, True):
            assert res.raw_column("string", 0, nullable) == ora.get_column("string", 0, nullable), f"nullable={nullable}"
        for fn in (tr.typed_column, tr.text_column):   # to_typed keeps ENUM as Value::String
            tc = fn(res, 0)
            assert tc.tag == tr.STRING
            assert np.array_equal(tc.valid, np.ones(n, bool) if valid is None else valid)
            for i in range(0, n, max(1, n // 97)):
                v = tc.value(i)
                if valid is None or valid[i]:
                    assert v.as_string().encode() == labels[idx[i]]
                else:
                    assert v.is_null()
        schema = res.get_schema()
        assert [f.type_id for f in schema.fields][0] == "string"


@pytest.mark.parametrize("n,k,max_len", [(5000, 3, 6), (70_001, 1000, 25), (4097, 66_000, 5)])
def test_enum_arrow_export_is_dictionary_encoded(ctx, n, k, max_len):
    batch, labels, idx, valid = _enum_batch(n, k, max_len, "ragged", 5 + k)
    with _result(ctx, batch) as res:
        arr = res.to_arrow(0)
        arr.validate(full=True)
        assert pa.types.is_dictionary(arr.type)
        assert arr.type.index_type == (pa.uint8() if k <= 256 else pa.uint16() if k <= 65536 else pa.uint32())
        assert arr.type.value_type == pa.string()
        assert arr.dictionary.to_pylist() == [x.decode() for x in labels]
        got_idx = np.asarray(arr.indices.fill_null(0))
        exp_idx = np.where(valid, idx, 0)
        assert np.array_equal(got_idx, exp_idx)           # NULL slots zeroed, like every fixed-width export
        assert arr.null_count == int((~valid).sum())
        exp = [labels[idx[i]].decode() if valid[i] else None for i in range(n)]
        assert arr.to_pylist() == exp
        rb = res.to_record_batch()
        rb.validate(full=True)
        assert rb.column(0).to_pylist() == exp
    del arr, rb  # exported arrays outlive the result: releasing them afterwards must be clean


def test_enum_index_past_the_dictionary_is_an_error(ctx):
    from duckdb_mbt_b200 import typed_result as tr
    from duckdb_mbt_b200.typed_result import DuckDBError
    counts = ch.chunk_counts(3000, "full")
    idx = np.zeros(3000, dtype=np.int64)
    idx[1234] = 9
    col = ch.enum_column("e", [b"a", b"bb", b"a-long-label-in-the-heap"], idx, counts)
    with _result(ctx, ch.ChunkBatch(counts, [col])) as res:
        with pytest.raises(DuckDBError, match="dictionary"):
            tr.text_column(res, 0)
        assert res.raw_column("string", 0) == b""     # getters never fail: empty Bytes (src/duckdb_native.c:2361-2368)


def test_enum_column_without_dictionary_is_rejected(ctx):
    from duckdb_mbt_b200 import arrow_result as ar
    from duckdb_mbt_b200 import native as nat
    counts = ch.chunk_counts(10, "full")
    col = ch.enum_column("e", [b"x"], np.zeros(10, np.int64), counts)
    col.dictionary = None
    with pytest.raises(Exception, match="dictionary"):
        ar.ArrowResult.from_chunks(ctx, ch.ChunkBatch(counts, [col]))
    assert "dictionary" in nat.last_error()


def test_enum_cells_through_connection_query_symbols(ctx):
    """Connection::query's per-cell loop (duckdb_mb_result_is_null / _value, src/duckdb_native.mbt:477-497) and the
    columnar string form give the labels; to_typed keeps them as Value::String (src/duckdb_parsing.mbt:119-122)."""
    from duckdb_mbt_b200 import native as nat
    from duckdb_mbt_b200.query_result import QueryResult, query_per_cell
    batch, labels, idx, valid = _enum_batch(5000, 6, 30, "ragged", 123)
    ora = oracle.OracleResult(batch)
    with _result(ctx, batch) as res:
        L, h = res.lib, res.handle
        assert L.duckdb_mb_result_column_type(h, 0) == ch.T_ENUM
        for r in range(0, 5000, 61):
            assert bool(L.duckdb_mb_result_is_null(h, 0, r)) == ora.cell_is_null(0, r) == (not valid[r])
            assert nat.moonbit_bytes(L.duckdb_mb_result_value(h, 0, r)) == ora.cell_value(0, r)
            if valid[r]:
                assert ora.cell_value(0, r) == labels[idx[r]]
        q = query_per_cell(res)
        c = QueryResult.from_result(res, q.column_types)
        assert c.rows == q.rows and c.nulls == q.nulls
        assert [row[0] for row in q.rows[:50]] == [labels[idx[i]].decode() if valid[i] else "" for i in range(50)]
        t = c.to_typed()
        first = int(np.argmax(valid))
        assert t.get_string(first, 0) == labels[idx[first]].decode()


def _expected_utf8(labels, idx, valid):
    """numpy restatement of what the Arrow utf8 form of an ENUM column holds: a valid row contributes its label, a NULL row nothing."""
    lens = np.array([len(x) for x in labels], dtype=np.int64)[idx]
    if valid is not None:
        lens = np.where(valid, lens, 0)
    offsets = np.zeros(len(idx) + 1, dtype=np.int64)
    np.cumsum(lens, out=offsets[1:])
    data = b"".join(labels[i] for i, v in zip(idx, valid if valid is not None else np.ones(len(idx), bool)) if v)
    return offsets, data


@pytest.mark.parametrize("n,k,max_len,pattern,null_frac", [
    (1, 1, 12, "full", 0.0), (2048, 2, 1, "full", 0.5), (2049, 256, 12, "ragged", 0.2),   # 256 labels: the largest fused dictionary
    (300_001, 7, 8, "ragged", 0.1), (1_000_000, 7, 7, "full", 0.0), (50_000, 3, 12, "ragged", 1.0)])
def test_enum_fused_lookup_and_pack_every_offset_and_byte(ctx, n, k, max_len, pattern, null_frac):
    """uint8 ENUM with labels of <= 12 bytes: indices -> utf8 in ONE launch (dmb_dev_enum_utf8: enum_pack_kernel<.., EW>),
    no string_t intermediate.  Every offset and every data byte against the numpy restatement and the oracle's cells."""
    from duckdb_mbt_b200 import typed_result as tr
    batch, labels, idx, valid = _enum_batch(n, k, max_len, pattern, 900 + n + k, null_frac=null_frac)
    if null_frac >= 1.0:
        assert not valid.any()
    exp_off, exp_data = _expected_utf8(labels, idx, valid)
    ora = oracle.OracleResult(batch)
    with _result(ctx, batch) as res:
        tc = tr.text_column(res, 0)
        assert np.array_equal(tc.offsets.astype(np.int64), exp_off)
        assert tc.data == exp_data
        assert np.array_equal(tc.valid, np.ones(n, bool) if valid is None else valid)
        for r in range(0, n, max(1, n // 53)):
            a, b = int(tc.offsets[r]), int(tc.offsets[r + 1])
            assert tc.data[a:b] == (b"" if ora.cell_is_null(0, r) else ora.cell_value(0, r))


def test_enum_fused_device_api_flags_long_labels_and_bad_indices(ctx):
    """dmb_dev_enum_utf8 at the device API: a label of > 12 bytes raises the heap-range flag, an index past the dictionary is counted
    and rendered empty, more than DMB_ENUM_FUSED_MAX_LABELS labels are refused before any launch."""
    import ctypes as C
    from duckdb_mbt_b200 import native as nat
    L = nat.lib()
    dev = torch.device("cuda")
    n, nch = 5000, 3
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def run(labels, idx_np, dict_size=None):
        d_offs, d_data = ch.enum_dict_arrays(labels)
        t_offs = torch.from_numpy(d_offs.view(np.uint8).copy()).to(dev)
        t_data = torch.from_numpy(np.concatenate([d_data, np.zeros(64, np.uint8)])).to(dev)
        slab = np.zeros(nch * 2048, np.uint8)
        slab[:n] = idx_np
        idx = torch.from_numpy(slab).to(dev)
        counts = torch.tensor([2048, 2048, n - 4096], dtype=torch.int32, device=dev)
        row_off = torch.tensor([0, 2048, 4096, n], dtype=torch.int64, device=dev)
        vecs = torch.tensor([[0, -1], [2048, -1], [4096, -1]], dtype=torch.int64, device=dev)
        bad = torch.zeros(1, dtype=torch.int64, device=dev)
        offsets = torch.zeros(4 * (n + 1) + 64, dtype=torch.uint8, device=dev)
        data = torch.zeros(12 * n + 64, dtype=torch.uint8, device=dev)
        total = torch.zeros(1, dtype=torch.int64, device=dev)
        scratch = torch.empty(L.dmb_dev_string_scratch_bytes(nch), dtype=torch.uint8, device=dev)
        ejob = nat.EnumJob(idx.data_ptr(), None, vecs.data_ptr(), None, t_offs.data_ptr(), t_data.data_ptr(), 1 << 41, bad.data_ptr(),
                           len(labels) if dict_size is None else dict_size, ch.P_U8)
        sjob = nat.StringJob(None, None, None, None, 0, 0, offsets.data_ptr(), data.data_ptr(), None, None, None, total.data_ptr(), 0, 0)
        rc = L.dmb_dev_enum_utf8(C.byref(ejob), C.byref(sjob), counts.data_ptr(), row_off.data_ptr(), nch, n, scratch.data_ptr(), stream)
        flags = L.dmb_dev_string_error(scratch.data_ptr(), stream) if rc == 0 else None
        tot = int(total.item())
        return rc, flags, int(bad.item()), offsets[:4 * (n + 1)].cpu().numpy().view("<i4"), bytes(data[:tot].cpu().numpy())

    rng = np.random.default_rng(4)
    labels = [b"a", b"", b"twelve bytes", b"xyz"]
    idx_np = rng.integers(0, 4, n).astype(np.uint8)
    rc, flags, nbad, off, dat = run(labels, idx_np)
    exp_off, exp_data = _expected_utf8(labels, idx_np, None)
    assert (rc, flags, nbad) == (0, 0, 0) and np.array_equal(off, exp_off) and dat == exp_data
    idx_bad = idx_np.copy()
    idx_bad[[7, 4999]] = 200
    rc, flags, nbad, off, dat = run(labels, idx_bad)
    assert (rc, flags, nbad) == (0, 0, 2)
    exp_off, exp_data = _expected_utf8(labels + [b""] * 252, idx_bad, None)   # rendered empty
    assert np.array_equal(off, exp_off) and dat == exp_data
    rc, flags, nbad, off, dat = run([b"a", b"thirteen byte"], (idx_np & 1))
    assert rc == 0 and flags != 0                                             # heap-range flag: a label the kernel cannot inline
    rc = run([b"a"], np.zeros(n, np.uint8), dict_size=257)[0]
    assert rc != 0 and "labels" in nat.last_error()


@pytest.mark.parametrize("phys,shift,large", [(ch.P_U8, 0, False), (ch.P_U8, 3, True), (ch.P_U16, 0, False), (ch.P_U16, 1, False),
                                              (ch.P_U32, 0, True), (ch.P_U32, 1, False)])
def test_enum_fused_device_api_index_widths_alignment_and_masks(ctx, phys, shift, large):
    """enum_pack_kernel at the device API: uint8 / uint16 / uint32 indices, vectors that start `shift` ELEMENTS past an aligned
    address (the thread's eight indices are then read one by one instead of as one vector), ragged chunks (a count that is not
    a multiple of 8, an empty chunk), validity masks with garbage indices under the NULL rows, int32 and int64 offsets."""
    import ctypes as C
    from duckdb_mbt_b200 import native as nat
    L = nat.lib()
    dev = torch.device("cuda")
    rng = np.random.default_rng(77 + phys + shift)
    np_t = {ch.P_U8: np.uint8, ch.P_U16: np.uint16, ch.P_U32: np.uint32}[phys]
    w = np.dtype(np_t).itemsize
    counts_np = np.array([2048, 2043, 0, 2048, 1, 777], dtype=np.uint32)
    nch, n = len(counts_np), int(counts_np.sum())
    labels = [b"", b"a", b"bc", b"twelve bytes", b"seven_7", b"0123456789", b"xyz"]
    k = len(labels)
    idx_np = rng.integers(0, k, n)
    valid = rng.random(n) >= 0.25
    # vector c sits `shift` elements behind slot c of the slab; rows past a chunk's count and rows under a NULL hold garbage
    slot = 2048 + 8
    slab = rng.integers(k, 250, nch * slot + 64).astype(np_t)
    masks = np.zeros((nch, 32), dtype=np.uint64)
    row_off = np.zeros(nch + 1, dtype=np.int64)
    np.cumsum(counts_np, out=row_off[1:])
    for c in range(nch):
        a, b = int(row_off[c]), int(row_off[c + 1])
        v = valid[a:b]
        vals = np.where(v, idx_np[a:b], rng.integers(k, 250, b - a)).astype(np_t)
        slab[c * slot + shift: c * slot + shift + (b - a)] = vals
        bits = np.zeros(2048, dtype=bool)
        bits[: b - a] = v
        bits[b - a:] = rng.random(2048 - (b - a)) > 0.5  # garbage past the count
        masks[c] = np.packbits(bits, bitorder="little").view(np.uint64)
    vecs_np = np.array([[(c * slot + shift) * w, c * 32] for c in range(nch)], dtype=np.int64)
    d_offs, d_data = ch.enum_dict_arrays(labels)
    t_offs = torch.from_numpy(d_offs.view(np.uint8).copy()).to(dev)
    t_data = torch.from_numpy(np.concatenate([d_data, np.zeros(64, np.uint8)])).to(dev)
    t_slab = torch.from_numpy(slab.view(np.uint8).copy()).to(dev)
    t_masks = torch.from_numpy(masks.view(np.uint8).reshape(-1).copy()).to(dev)
    t_counts = torch.from_numpy(counts_np.view(np.uint8).copy()).to(dev)
    t_row_off = torch.from_numpy(row_off.view(np.uint8).copy()).to(dev)
    t_vecs = torch.from_numpy(vecs_np.view(np.uint8).reshape(-1).copy()).to(dev)
    bad = torch.zeros(1, dtype=torch.int64, device=dev)
    ow = 8 if large else 4
    offsets = torch.zeros(ow * (n + 1) + 64, dtype=torch.uint8, device=dev)
    data = torch.zeros(12 * n + 64, dtype=torch.uint8, device=dev)
    total = torch.zeros(1, dtype=torch.int64, device=dev)
    scratch = torch.empty(L.dmb_dev_string_scratch_bytes(nch), dtype=torch.uint8, device=dev)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    ejob = nat.EnumJob(t_slab.data_ptr(), t_masks.data_ptr(), t_vecs.data_ptr(), None, t_offs.data_ptr(), t_data.data_ptr(), 1 << 41,
                       bad.data_ptr(), k, phys)
    mode = 1 if large else 0  # DMB_STR_ARROW_LARGE / DMB_STR_ARROW_UTF8
    sjob = nat.StringJob(None, None, None, None, 0, 0, offsets.data_ptr(), data.data_ptr(), None, None, None, total.data_ptr(), mode, 0)
    rc = L.dmb_dev_enum_utf8(C.byref(ejob), C.byref(sjob), t_counts.data_ptr(), t_row_off.data_ptr(), nch, n, scratch.data_ptr(), stream)
    assert rc == 0, nat.last_error()
    assert L.dmb_dev_string_error(scratch.data_ptr(), stream) == 0, nat.last_error()
    assert int(bad.item()) == 0  # garbage under NULL rows is never counted
    exp_off, exp_data = _expected_utf8(labels, idx_np, valid)
    got_off = offsets[: ow * (n + 1)].cpu().numpy().view("<i8" if large else "<i4").astype(np.int64)
    assert np.array_equal(got_off, exp_off)
    assert int(total.item()) == len(exp_data)
    assert bytes(data[: len(exp_data)].cpu().numpy()) == exp_data
