"""CPU-only: the layout the reverse LIST path writes (Arrow list -> DuckDB LIST vectors), restated in numpy and held to
pyarrow's own reading of the arrays (`to_pylist`), and the appender's sub-batch cut (`dmb_rev_list_cut`) pinned.

The restatement is what tests/test_gpu_append_list.py compares the device with: per row a duckdb_list_entry
{off[r] - off[first row of r's chunk], off[r+1] - off[r]} (length 0 for a NULL row), 32 list-mask words per 2048-row
chunk, and per chunk a child mask that starts at bit 0 of that chunk's first element."""
import ctypes as C

import numpy as np
import pytest

pa = pytest.importorskip("pyarrow")

VEC = 2048


def bits_of(arr_bitmap_buf, bit_offset: int, n: int) -> np.ndarray:
    """bool per position of an Arrow bitmap (None = all valid)"""
    if arr_bitmap_buf is None:
        return np.ones(n, dtype=bool)
    raw = np.frombuffer(arr_bitmap_buf, dtype=np.uint8)
    return np.unpackbits(raw, bitorder="little")[bit_offset: bit_offset + n].astype(bool)


def words_of(valid: np.ndarray, nwords: int) -> np.ndarray:
    """LSB-first uint64 words of a bool array, zero past its end"""
    out = np.zeros(nwords * 8, dtype=np.uint8)
    packed = np.packbits(valid.astype(np.uint8), bitorder="little")
    out[: packed.shape[0]] = packed
    return out.view(np.uint64)


def rev_list_reference(offsets: np.ndarray, parent_valid: np.ndarray, child_valid: np.ndarray):
    """offsets: the n + 1 Arrow offsets of the slice; parent_valid: n bools; child_valid: the bools of Arrow elements
    [offsets[0], offsets[n]).  Returns (entries [nch*2048, 2] uint64, list masks [nch*32], child masks (concatenated),
    child_word [nch + 1], null count)."""
    off = np.asarray(offsets, dtype=np.int64)
    n = off.shape[0] - 1
    nch = (n + VEC - 1) // VEC
    rows = np.arange(n)
    base = off[(rows // VEC) * VEC]
    lens = off[1:] - off[:-1]
    entries = np.zeros((nch * VEC, 2), dtype=np.uint64)
    entries[:n, 0] = (off[:-1] - base).astype(np.uint64)
    entries[:n, 1] = np.where(parent_valid, lens, 0).astype(np.uint64)
    masks = np.concatenate([words_of(parent_valid[k * VEC:(k + 1) * VEC], 32) for k in range(nch)]) if nch else np.zeros(0, np.uint64)
    child_word = np.zeros(nch + 1, dtype=np.int64)
    cwords = []
    for k in range(nch):
        e0, e1 = off[k * VEC] - off[0], off[min((k + 1) * VEC, n)] - off[0]
        nw = (e1 - e0 + 63) // 64
        cwords.append(words_of(child_valid[e0:e1], nw))
        child_word[k + 1] = child_word[k] + nw
    child_masks = np.concatenate(cwords) if cwords else np.zeros(0, np.uint64)
    return entries, masks, child_masks, child_word, int(n - parent_valid.sum())


def arrow_parts(arr):
    """(offsets of the slice, parent valid, child valid from the slice's first element, child values) of a pyarrow
    list array, read from its buffers the way the appender reads them"""
    n = len(arr)
    bufs = arr.buffers()
    odt = np.int64 if pa.types.is_large_list(arr.type) else np.int32
    off = np.frombuffer(bufs[1], dtype=odt)[arr.offset: arr.offset + n + 1].astype(np.int64)
    parent_valid = bits_of(bufs[0] if arr.null_count else None, arr.offset, n)
    child = arr.values
    cbufs = child.buffers()
    cvalid_all = bits_of(cbufs[0] if child.null_count else None, child.offset, len(child))
    return off, parent_valid, cvalid_all[off[0]: off[-1]], child.to_pylist()[off[0]: off[-1]]


def decode(entries, masks, child_masks, child_word, off, child_values, n):
    """the restated vectors read back as DuckDB would: per chunk, entries index that chunk's own child vector"""
    out = []
    for r in range(n):
        k = r // VEC
        if not (int(masks[k * 32 + (r % VEC) // 64]) >> (r % 64)) & 1:
            out.append(None)
            continue
        o, ln = int(entries[r, 0]), int(entries[r, 1])
        e0 = int(off[k * VEC] - off[0])
        size = int(off[min((k + 1) * VEC, n)] - off[k * VEC])
        assert o + ln <= size
        row = []
        for j in range(o, o + ln):
            bit = (int(child_masks[child_word[k] + j // 64]) >> (j % 64)) & 1
            row.append(child_values[e0 + j] if bit else None)
        out.append(row)
    return out


def make_list_array(n, seed, large=False, child_off=0, null_frac=0.2, child_null_frac=0.15, max_len=7, empty_frac=0.1):
    """a list<int32> / large_list<int32> with NULL rows over non-empty segments, empty lists and a child array that
    starts `child_off` elements into its buffers"""
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, max_len + 1, n)
    lens[rng.random(n) < empty_frac] = 0
    off = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    total = int(off[-1])
    vals = rng.integers(-2**31, 2**31, total + child_off, dtype=np.int64).astype(np.int32)
    cmask = rng.random(total + child_off) < child_null_frac
    child = pa.array(vals, mask=cmask).slice(child_off)
    mask = pa.array(rng.random(n) < null_frac)
    typ = pa.LargeListArray if large else pa.ListArray
    return typ.from_arrays(pa.array(off, pa.int64() if large else pa.int32()), child, mask=mask)


@pytest.mark.parametrize("n,large,child_off,slice_", [
    (1, False, 0, None), (7, True, 3, None), (2048, False, 5, None), (2049, True, 0, (1, 2047)),
    (10_000, False, 11, (5, 9_000)), (6_000, True, 1, (2047, 3_000)), (300, False, 0, (64, 100))])
def test_reference_agrees_with_pyarrow(n, large, child_off, slice_):
    arr = make_list_array(n, n + child_off, large, child_off)
    if slice_:
        arr = arr.slice(*slice_)
    off, pv, cv, cvals = arrow_parts(arr)
    ent, masks, cmasks, cword, nulls = rev_list_reference(off, pv, cv)
    assert nulls == arr.null_count
    assert decode(ent, masks, cmasks, cword, off, cvals, len(arr)) == arr.to_pylist()
    # a NULL row owns no elements even where Arrow gives it a segment
    assert not np.any(ent[: len(arr), 1][~pv])
    assert np.any((off[1:] - off[:-1])[~pv] > 0) or pv.all()


def test_reference_all_empty_lists():
    arr = pa.ListArray.from_arrays(pa.array(np.zeros(5001, np.int32)), pa.array([], pa.int32()))
    off, pv, cv, cvals = arrow_parts(arr)
    ent, masks, cmasks, cword, nulls = rev_list_reference(off, pv, cv)
    assert cmasks.shape[0] == 0 and not cword.any() and not ent.any() and nulls == 0
    assert decode(ent, masks, cmasks, cword, off, cvals, len(arr)) == arr.to_pylist()


def test_reference_chunk_child_masks_start_at_bit_zero():
    # chunk sizes that are not multiples of 64: chunk 1's mask is the dense bitmap shifted by chunk 0's size
    lens = np.full(2 * VEC, 1)
    lens[0] = 0  # chunk 0: 2047 elements
    off = np.concatenate([[0], np.cumsum(lens)])
    cv = np.arange(off[-1]) % 3 != 0
    _, _, cmasks, cword, _ = rev_list_reference(off, np.ones(2 * VEC, bool), cv)
    assert list(cword) == [0, 32, 64]
    assert np.array_equal(np.unpackbits(cmasks[32:64].view(np.uint8), bitorder="little")[:VEC].astype(bool), cv[2047:2047 + VEC])
    assert int(cmasks[31]) >> 63 == 0  # bit 2047 of chunk 0's mask is past its 2047 elements


# ------------------------------------------------------------------------------------------- the sub-batch cut
def _cut(bounds_per_list, max_chunks, cap):
    """all sub-batches [k0, k1) of a batch through the library's dmb_rev_list_cut"""
    import __graft_entry__ as g
    g.build()
    from duckdb_mbt_b200 import native as nat
    L = nat.lib()
    arrays = [np.ascontiguousarray(b, dtype=np.int64) for b in bounds_per_list]
    ptrs = (C.c_void_p * max(len(arrays), 1))(*[a.ctypes.data for a in arrays])
    nch = (len(arrays[0]) - 1) if arrays else 0
    cuts, k0 = [], 0
    while k0 < nch:
        k1 = L.dmb_rev_list_cut(C.cast(ptrs, C.c_void_p), len(arrays), nch, k0, max_chunks, cap)
        cuts.append((k0, k1))
        k0 = k1
    return cuts


def test_cut_on_chunk_boundaries_by_rows():
    bounds = np.arange(11) * 100  # 10 chunks of 100 elements
    assert _cut([bounds], 4, 10**9) == [(0, 4), (4, 8), (8, 10)]


def test_cut_by_child_element_cap():
    bounds = np.arange(11) * 100
    # 250 elements per sub-batch at most: two chunks each
    assert _cut([bounds], 100, 250) == [(0, 2), (2, 4), (4, 6), (6, 8), (8, 10)]
    # the tightest of several LIST columns decides
    other = np.concatenate([[0], np.cumsum([10, 10, 10, 500, 10, 10, 10, 10, 10, 10])])
    assert _cut([bounds, other], 100, 520) == [(0, 3), (3, 6), (6, 10)]


def test_cut_keeps_a_chunk_larger_than_the_cap_whole():
    bounds = np.concatenate([[0], np.cumsum([5, 5, 10**6, 5, 5])])
    cuts = _cut([bounds], 100, 1000)
    assert cuts == [(0, 2), (2, 3), (3, 5)]
    assert all(k1 > k0 for k0, k1 in cuts)
