"""CPU: what an ENUM column holds after an Arrow array is appended to it (a plain-Python restatement of the contract in
include/duckdb_mb_gpu.h, dmb_rev_enum_job / duckdb_mb_gpu_appender_set_enum), checked against hand-written answers; and
the host side of the label lookup (dmb_rev_enum_table / dmb_rev_enum_lookup, the probe the device runs) at table sizes
small enough to force collisions."""
import ctypes as C

import numpy as np
import pytest

pa = pytest.importorskip("pyarrow")


def _label_bytes(v):
    return v.encode("utf-8") if isinstance(v, str) else bytes(v)


def enum_reference(arr, labels):
    """(positions int64[n], validity bool[n], first offending row or None) of `arr` appended to an ENUM of `labels`.
    Read through pyarrow's own decoding: a NULL row (by the Arrow validity) is NULL whatever sits under it; a valid row
    whose dictionary entry is NULL is NULL; a valid row whose label is not an ENUM label, or whose index is outside the
    dictionary, is an error.  Labels match byte-exactly."""
    pos_of = {_label_bytes(x): i for i, x in enumerate(labels)}
    n = len(arr)
    pos = np.zeros(n, np.int64)
    valid = np.zeros(n, bool)
    first = None
    if pa.types.is_dictionary(arr.type):
        entries = [None if v is None else _label_bytes(v) for v in arr.dictionary.to_pylist()]
        rows = arr.indices.to_pylist()
    else:
        entries = None
        rows = arr.to_pylist()
    for i, v in enumerate(rows):
        if v is None:
            continue
        if entries is not None:
            if v < 0 or v >= len(entries):
                first = i if first is None else first
                continue
            v = entries[v]
            if v is None:
                continue
        p = pos_of.get(_label_bytes(v))
        if p is None:
            first = i if first is None else first
            continue
        pos[i], valid[i] = p, True
    return pos, valid, first


def dictionary_array(indices, index_type, dictionary, mask=None):
    """a DictionaryArray whose indices are taken as given (out-of-range ones included, under NULL rows or not)"""
    ind = pa.array(np.asarray(indices), type=index_type, mask=None if mask is None else np.asarray(mask))
    return pa.DictionaryArray.from_arrays(ind, dictionary, safe=False)


# ------------------------------------------------------------------------------------------- the reference, by hand
LABELS = ["AIR", "MAIL", "SHIP", ""]


def test_reference_on_strings():
    arr = pa.array(["SHIP", None, "", "AIR", "MAIL", "ship"])
    pos, valid, first = enum_reference(arr, LABELS)
    assert valid.tolist() == [True, False, True, True, True, False]
    assert pos.tolist() == [2, 0, 3, 0, 1, 0]
    assert first == 5  # "ship": no case folding


def test_reference_null_dictionary_entries_and_unused_entries():
    d = pa.array(["MAIL", None, "TRUCK", "AIR"])  # TRUCK is not a label but no valid row uses it
    arr = dictionary_array([0, 1, 3, 0, 1], pa.int8(), d)
    pos, valid, first = enum_reference(arr, LABELS)
    assert valid.tolist() == [True, False, True, True, False]
    assert pos.tolist() == [1, 0, 0, 1, 0]
    assert first is None


def test_reference_ignores_garbage_under_null_rows():
    d = pa.array(["AIR", "SHIP"])
    arr = dictionary_array([1, -5, 99, 0], pa.int16(), d, mask=[False, True, True, False])
    pos, valid, first = enum_reference(arr, LABELS)
    assert valid.tolist() == [True, False, False, True]
    assert pos.tolist() == [2, 0, 0, 0]
    assert first is None


def test_reference_duplicate_dictionary_entries_map_to_one_label():
    d = pa.array(["SHIP", "AIR", "SHIP"])
    arr = dictionary_array([0, 2, 1], pa.uint8(), d)
    pos, valid, _ = enum_reference(arr, LABELS)
    assert pos.tolist() == [2, 2, 0] and valid.all()


def test_reference_errors_name_the_first_offending_row():
    d = pa.array(["AIR", "RAIL"])
    assert enum_reference(dictionary_array([0, 0, 1, 0], pa.int32(), d), LABELS)[2] == 2  # a label the ENUM lacks
    assert enum_reference(dictionary_array([0, 2, 1], pa.int64(), d), LABELS)[2] == 1     # index past the dictionary
    assert enum_reference(dictionary_array([0, -1], pa.int8(), d), LABELS)[2] == 1        # negative index
    assert enum_reference(pa.array(["AIR", "AIR ", None]), LABELS)[2] == 1                # no trimming


# ------------------------------------------------------------------------------------------- the host lookup table
@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from duckdb_mbt_b200 import native as nat
    return nat.lib()


def _table(lib, labels, size):
    from duckdb_mbt_b200 import appender as ap
    from duckdb_mbt_b200 import native as nat
    d, keep = ap.enum_dict(labels)
    slots = C.create_string_buffer(size * nat.ENUM_SLOT_BYTES)
    ok = lib.dmb_rev_enum_table(C.byref(d), size, slots)
    return ok, (d, keep, slots)


def _lookup(lib, t, b: bytes):
    d, _, slots = t
    buf = C.create_string_buffer(b, len(b) + 1)
    return lib.dmb_rev_enum_lookup(slots, len(slots) // 32, C.byref(d), buf, len(b))


NEAR = [b"a", b"ab", b"abc", b"", b"x" * 12, b"x" * 13, b"prefix_0000_mid_tail", "café crème brûlée".encode()]


@pytest.mark.parametrize("size", [16, 32, 1024])
def test_every_label_is_found_at_its_position_even_in_a_crowded_table(lib, size):
    ok, t = _table(lib, NEAR, size)
    assert ok
    for i, x in enumerate(NEAR):
        assert _lookup(lib, t, x) == i


def test_a_table_with_one_free_slot_still_finds_everything(lib):
    labels = [b"l%d" % i for i in range(15)]
    ok, t = _table(lib, labels, 16)  # 15 labels in 16 slots: chains run through most of the table
    assert ok
    assert [_lookup(lib, t, x) for x in labels] == list(range(15))
    assert _lookup(lib, t, b"l15") == -1


@pytest.mark.parametrize("probe", [b"abcd", b"a\0", b"ab\0", b"A", b" a", b"x" * 11, b"x" * 14, b"prefix_0000_MID_tail",
                                   b"prefix_0000_mid_tai", b"prefix_0000_mid_tailx", "café crème brûléE".encode()])
def test_prefixes_extensions_and_near_misses_are_not_found(lib, probe):
    ok, t = _table(lib, NEAR, 16)
    assert ok
    assert _lookup(lib, t, probe) == -1


def test_long_labels_that_differ_only_in_the_middle(lib):
    labels = [b"0123456789ab" + bytes([c]) * 40 + b"TAIL" for c in range(65, 91)]
    ok, t = _table(lib, labels, 32)
    assert ok
    assert [_lookup(lib, t, x) for x in labels] == list(range(26))
    assert _lookup(lib, t, b"0123456789ab" + b"A" * 39 + b"B" + b"TAIL") == -1


def test_duplicate_labels_and_small_tables_are_refused(lib):
    from duckdb_mbt_b200 import native as nat
    ok, _ = _table(lib, [b"a", b"b", b"a"], 16)
    assert not ok and "both 'a'" in nat.last_error()
    ok, _ = _table(lib, [b"a", b"b", b"c", b"d"], 4)
    assert not ok and "cannot hold" in nat.last_error()
    ok, _ = _table(lib, [b"a", b"b"], 12)
    assert not ok
