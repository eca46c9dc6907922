"""Arrow string views and dictionary-encoded strings appended to VARCHAR / BLOB columns: the case builders that
tests/test_gpu_append_strings.py uses, checked without a GPU.

What DuckDB holds after such an append is what it holds for the same array cast to utf8 / binary, so
tests/reverse_semantics.py must give views and dictionaries the same cells as their casts.  The builders must really
produce what the GPU tests rely on: views spread over several data buffers, garbage in inline padding and under NULL
rows, and every edge value at every placement (chunk rows 0 and 2047, the first and last rows of a 4096-row sub-batch,
Arrow offsets 0-7)."""
import struct

import numpy as np
import pytest

pa = pytest.importorskip("pyarrow")

import reverse_semantics as rs  # noqa: E402
from duckdb_mbt_b200 import chunks as ch  # noqa: E402
from test_rev_enum_cpu import dictionary_array  # noqa: E402

SUB_ROWS = 4096  # DMB_REV_BATCH_ROWS of the GPU tests
PLACES = (0, 2047, 2048, SUB_ROWS - 1, SUB_ROWS, SUB_ROWS + 2047)  # chunk and sub-batch edges


def edge_values() -> list:
    """lengths 0-16 and 70 KB, exactly 12 and 13, NUL bytes, UTF-8 across byte 12"""
    out = [bytes(range(97, 97 + k)) for k in range(17)]
    out += [b"\x00" * 12, b"a\x00b\x00c\x00d\x00e\x00f\x00g", b"x" * 70_000, "abcdefghijkéz".encode(), "0123456789€".encode(),
            ("é" * 8).encode()]
    return out


def _bits(valid: np.ndarray) -> bytes:
    return np.packbits(valid.astype(np.uint8), bitorder="little").tobytes() + b"\x00" * 8


def view_array(values: list, binary: bool = False, nbufs: int = 3, seed: int = 0):
    """a utf8_view (binary_view) array of `values` (bytes or None) built from its buffers: pointer views spread round-robin
    over `nbufs` data buffers with gaps between strings, random garbage in the inline padding and in NULL rows' views"""
    rng = np.random.default_rng(seed)
    n = len(values)
    views = rng.integers(0, 256, 16 * n, dtype=np.uint8)
    bufs = [bytearray(rng.integers(0, 256, 5, dtype=np.uint8).tobytes()) for _ in range(nbufs)]
    valid = np.asarray([v is not None for v in values])
    for i, v in enumerate(values):
        if v is None:
            continue
        if len(v) <= 12:
            views[16 * i:16 * i + 4] = np.frombuffer(struct.pack("<i", len(v)), np.uint8)
            views[16 * i + 4:16 * i + 4 + len(v)] = np.frombuffer(v, np.uint8)  # padding past len stays garbage
        else:
            b = i % nbufs
            off = len(bufs[b])
            bufs[b] += v + bytes(int(rng.integers(0, 4)))
            views[16 * i:16 * i + 16] = np.frombuffer(struct.pack("<i4sii", len(v), v[:4], b, off), np.uint8)
    typ = pa.binary_view() if binary else pa.string_view()
    buffers = [pa.py_buffer(_bits(valid)), pa.py_buffer(views.tobytes())] + [pa.py_buffer(bytes(b)) for b in bufs]
    return pa.Array.from_buffers(typ, n, buffers, null_count=int((~valid).sum()))


def plain(values: list, binary: bool = False):
    """the utf8 (binary) array of `values`: what a view or dictionary array of them is cast to.  (pyarrow's own cast
    reads the garbage view_array leaves in inline padding, which Arrow's validation rejects, so it is not used.)"""
    return pa.array([v if v is None or binary else v.decode() for v in values], pa.binary() if binary else pa.string())


def raw_views(arr) -> np.ndarray:
    """the 16-byte views of a view array's slice as an (n, 16) uint8 array"""
    buf = np.frombuffer(arr.buffers()[1], np.uint8)
    return buf[16 * arr.offset:16 * (arr.offset + len(arr))].reshape(-1, 16)


def placed(values: list, n: int, rng, nulls: float = 0.1) -> list:
    """n cells: every edge value at every place in PLACES (each place shifts through the edges), the rest random edges
    and NULLs"""
    out = [values[int(k)] for k in rng.integers(0, len(values), n)]
    for i in np.nonzero(rng.random(n) < nulls)[0]:
        out[i] = None
    for p, at in enumerate(PLACES):
        for e in range(len(values)):
            r = at + e * (2 * SUB_ROWS + 2048) if at + e * (2 * SUB_ROWS + 2048) < n else None
            if r is not None:
                out[r] = values[(e + p) % len(values)]
    return out


def n_for(values: list) -> int:
    return len(values) * (2 * SUB_ROWS + 2048) + 4


# ------------------------------------------------------------------------------------------- the semantics
@pytest.mark.parametrize("binary", [False, True])
def test_views_have_the_cells_of_their_casts(binary):
    vals = edge_values() + [None]
    arr = view_array(vals, binary=binary, nbufs=3, seed=1)
    with pytest.raises(pa.ArrowInvalid, match="padding"):  # the garbage is there
        arr.validate(full=True)
    t = ch.T_BLOB if binary else ch.T_VARCHAR
    exp = rs.expected_cells(plain(vals, binary), t)
    assert rs.expected_cells(arr, t) == exp == [None if v is None else v for v in vals]


def test_dictionaries_have_the_cells_of_their_casts():
    d = pa.array([b"x" * 20, None, b"short", b""], pa.binary())
    arr = dictionary_array([0, 1, 2, 3, 9, 2], pa.int8(), d, mask=[False, False, False, False, True, False])
    assert rs.expected_cells(arr, ch.T_BLOB) == [b"x" * 20, None, b"short", b"", None, b"short"]
    assert rs.expected_cells(arr.slice(2), ch.T_BLOB) == rs.expected_cells(arr.cast(pa.binary()).slice(2), ch.T_BLOB)
    sd = pa.array(["a", "bb", None, "c" * 13]).slice(1)
    arr = dictionary_array([0, 1, 2], pa.uint16(), sd)
    assert rs.expected_cells(arr, ch.T_VARCHAR) == [b"bb", None, b"c" * 13]


# ------------------------------------------------------------------------------------------- the builders
def test_view_builder_spreads_buffers_and_leaves_garbage():
    vals = edge_values() * 3 + [None] * 5
    arr = view_array(vals, nbufs=3, seed=2)
    assert arr.to_pylist() == [None if v is None else v.decode() for v in vals]
    assert len(arr.buffers()) == 5  # validity, views, three data buffers
    v = raw_views(arr)
    lens = v[:, :4].copy().view(np.int32)[:, 0]
    idx = v[:, 8:12].copy().view(np.int32)[:, 0]
    valid = np.asarray([x is not None for x in vals])
    assert set(idx[valid & (lens > 12)]) == {0, 1, 2}
    inline = valid & (lens < 12)
    pad_garbage = [v[i, 4 + lens[i]:].any() for i in np.nonzero(inline)[0]]
    assert sum(pad_garbage) > len(pad_garbage) // 2
    assert v[~valid].any()  # NULL rows' views are garbage


def test_placement_puts_every_edge_at_every_place():
    vals = edge_values()
    n = n_for(vals)
    cells = placed(vals, n, np.random.default_rng(3))
    for p, at in enumerate(PLACES):
        got = {cells[at + e * (2 * SUB_ROWS + 2048)] for e in range(len(vals))}
        assert got == set(vals), at
    assert {at % 2048 for at in PLACES} == {0, 2047}  # chunk rows 0 / 2047
    assert {0, SUB_ROWS - 1, SUB_ROWS} <= set(PLACES)  # a sub-batch's first and last rows


def test_offsets_slice_views_and_keep_16_byte_alignment_of_each_view():
    vals = edge_values()
    base = view_array(vals + vals, seed=4)
    for off in range(8):
        s = base.slice(off, len(vals))
        assert s.offset == off
        assert s.to_pylist() == [v.decode() for v in (vals + vals)[off:off + len(vals)]]
        assert raw_views(s).shape == (len(vals), 16)
