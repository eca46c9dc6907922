"""STRUCT columns on the appender's reverse path, restated in plain pyarrow / numpy (no GPU).

`struct_contract` is what DuckDB holds after an Arrow struct array is appended to a STRUCT column: the struct's mask is
its own bitmap ANDed with those of its ancestor structs, and a field is NULL wherever it is NULL itself or an ancestor
struct row is NULL.  Fields are read at the struct's offset plus their own (the Arrow C data interface does not apply a
struct's offset to its children).  It is checked against hand-written answers and against pyarrow's
`StructArray.flatten()`, which applies both the offset and the parent NULLs.

`mask_and` restates rev_mask_kernel (L0 dmb_dev_rev_mask_batch): two bitmaps at their own bit offsets ANDed into whole
2048-row chunks of 64-bit words from an output bit offset on, every other bit zero.  It is checked bit by bit against a
loop over the rows."""
import numpy as np
import pytest

pa = pytest.importorskip("pyarrow")

VECTOR_SIZE = 2048


def _valid(arr) -> np.ndarray:
    return np.asarray(arr.is_valid().to_numpy(zero_copy_only=False), dtype=bool)


def struct_contract(arr, ancestors=None, path=()) -> dict:
    """`arr` (a pyarrow StructArray, sliced or not) -> {path: (mask, field array)}: path () is the struct itself (array
    None), (i,) its field i, (i, j) field j of a STRUCT field i, ...  The field array has the struct's slice applied and
    only its own NULLs; the mask is what the appended vector holds."""
    valid = _valid(arr) if ancestors is None else ancestors & _valid(arr)
    out = {path: (valid, None)}
    for i in range(arr.type.num_fields):
        f = arr.field(i)  # the struct's offset applied, its NULLs not
        if pa.types.is_struct(f.type):
            out.update(struct_contract(f, valid, path + (i,)))
        else:
            out[path + (i,)] = (valid & _valid(f), f)
    return out


def flatten_reference(arr, path=()) -> dict:
    """the same masks and values read through StructArray.flatten()"""
    out = {path: (_valid(arr), None)}
    for i, f in enumerate(arr.flatten()):
        if pa.types.is_struct(f.type):
            out.update(flatten_reference(f, path + (i,)))
        else:
            out[path + (i,)] = (_valid(f), f)
    return out


def mask_and(a: bytes, a_off: int, b: bytes, b_off: int, nrows: int, out_off: int) -> np.ndarray:
    """rev_mask_kernel's output words: bits out_off .. out_off + nrows - 1 are row r's `a AND b` (None: all valid)"""
    nwords = ((out_off + nrows + VECTOR_SIZE - 1) // VECTOR_SIZE) * 32
    bits = np.zeros(nwords * 64, dtype=bool)
    ra = np.unpackbits(np.frombuffer(a, np.uint8), bitorder="little")[a_off:a_off + nrows].astype(bool) if a is not None else True
    rb = np.unpackbits(np.frombuffer(b, np.uint8), bitorder="little")[b_off:b_off + nrows].astype(bool) if b is not None else True
    bits[out_off:out_off + nrows] = np.ones(nrows, bool) & ra & rb
    return np.packbits(bits, bitorder="little").view(np.uint64)


def _mask_and_loop(a, a_off, b, b_off, nrows, out_off) -> np.ndarray:
    nwords = ((out_off + nrows + VECTOR_SIZE - 1) // VECTOR_SIZE) * 32
    words = [0] * nwords
    bit = lambda buf, i: buf is None or (buf[i >> 3] >> (i & 7)) & 1  # noqa: E731
    for r in range(nrows):
        if bit(a, a_off + r) and bit(b, b_off + r):
            p = out_off + r
            words[p >> 6] |= 1 << (p & 63)
    return np.array(words, dtype=np.uint64)


# ---------------------------------------------------------------------------------------------- the contract
def _nested(rng, n, lead):
    """STRUCT<i int32, b bool, s utf8, inner STRUCT<x int64, inner2 STRUCT<y bool>>> of n rows after `lead` rows, NULLs at
    every level, every field sliced from a longer array"""
    def ints(m, t):
        return pa.array(rng.integers(-1000, 1000, m).astype(t), mask=rng.random(m) < 0.2)

    def bools(m):
        return pa.array(rng.random(m) < 0.5, mask=rng.random(m) < 0.2)

    m = n + lead
    y = bools(m + 5).slice(5)
    inner2 = pa.StructArray.from_arrays([y], names=["y"], mask=pa.array(rng.random(m) < 0.2))
    x = ints(m + 3, np.int64).slice(3)
    inner = pa.StructArray.from_arrays([x, inner2], names=["x", "inner2"], mask=pa.array(rng.random(m) < 0.2)).slice(1)
    i = ints(m + 2, np.int32).slice(1)[:m - 1]
    b = bools(m + 7).slice(7)[:m - 1]
    s = pa.array([None if rng.random() < 0.2 else "v%d" % k * (k % 5) for k in range(m - 1)])
    return pa.StructArray.from_arrays([i, b, s, inner], names=["i", "b", "s", "inner"],
                                      mask=pa.array(rng.random(m - 1) < 0.15)).slice(lead - 1, n)


def test_contract_by_hand():
    # the issue's shape: a field with an offset of its own, the struct sliced on top
    c = pa.array([10, 11, 12, 13, 14, 15, 16], pa.int32())
    b = pa.array([True, None, False, True, False], pa.bool_())
    st = pa.StructArray.from_arrays([c.slice(2), b], names=["c", "b"], mask=pa.array([False, True, False, False, True])).slice(1, 4)
    got = struct_contract(st)
    assert got[()][0].tolist() == [False, True, True, False]
    assert got[(0,)][0].tolist() == [False, True, True, False]
    assert got[(0,)][1].to_pylist() == [13, 14, 15, 16]  # field row = field offset 2 + struct offset 1 + i
    assert got[(1,)][0].tolist() == [False, True, True, False]  # its own NULL (row 0) lies under a NULL struct row
    assert got[(1,)][1].to_pylist() == [None, False, True, False]
    # nested: an inner NULL struct row hides its field, an outer one hides both
    y = pa.array([True, True, None, True])
    inner = pa.StructArray.from_arrays([y], names=["y"], mask=pa.array([False, True, False, False]))
    outer = pa.StructArray.from_arrays([inner], names=["inner"], mask=pa.array([False, False, False, True]))
    got = struct_contract(outer)
    assert got[()][0].tolist() == [True, True, True, False]
    assert got[(0,)][0].tolist() == [True, False, True, False]
    assert got[(0, 0)][0].tolist() == [True, False, False, False]


@pytest.mark.parametrize("lead", [1, 2, 5, 8])
def test_contract_matches_flatten(lead):
    rng = np.random.default_rng(lead)
    st = _nested(rng, 3000, lead)
    got, ref = struct_contract(st), flatten_reference(st)
    assert got.keys() == ref.keys()
    for path, (valid, arr) in got.items():
        assert valid.tolist() == ref[path][0].tolist(), path
        if arr is not None:  # the values under a valid row; flatten's payload under NULL rows is not defined
            vals, rvals = arr.to_pylist(), ref[path][1].to_pylist()
            assert [v for v, ok in zip(vals, valid) if ok] == [v for v, ok in zip(rvals, valid) if ok], path


def test_field_array_is_not_the_reference():
    """StructArray.field applies the slice but not the struct's NULLs: the contract masks it"""
    st = pa.StructArray.from_arrays([pa.array([1, 2, 3])], names=["a"], mask=pa.array([False, True, False]))
    assert st.field(0).to_pylist() == [1, 2, 3]
    assert struct_contract(st)[(0,)][0].tolist() == [True, False, True]


# ---------------------------------------------------------------------------------------------- L0 restatement
NROWS = [0, 1, 63, 64, 65, 2047, 2048, 2049, 4096 + 2049]


@pytest.mark.parametrize("nrows", NROWS)
def test_mask_and_at_every_bit_offset(nrows):
    rng = np.random.default_rng(nrows)
    a = rng.integers(0, 256, (nrows + 64) // 8 + 9, dtype=np.uint8).tobytes()
    b = rng.integers(0, 256, (nrows + 64) // 8 + 9, dtype=np.uint8).tobytes()
    for off in range(64):
        a_off, b_off, out_off = off, (off * 37) % 64, off % 8
        got = mask_and(a, a_off, b, b_off, nrows, out_off)
        assert np.array_equal(got, _mask_and_loop(a, a_off, b, b_off, nrows, out_off)), off
    for ab in ((None, b), (a, None), (None, None)):
        assert np.array_equal(mask_and(ab[0], 3, ab[1], 5, nrows, 0), _mask_and_loop(ab[0], 3, ab[1], 5, nrows, 0))
