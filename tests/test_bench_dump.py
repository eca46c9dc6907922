"""bench.py --dump-outputs: the arrays written for a step are the step's Arrow buffers at the sampled rows, in float32 /
float64, and the same step gives the same files.  CPU only: the step's buffers are host tensors here."""
import os
from types import SimpleNamespace

import numpy as np
import pytest

torch = pytest.importorskip("torch")

import bench  # noqa: E402
from duckdb_mbt_b200 import chunks as ch  # noqa: E402


def _as_u8(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy())


def test_dump_step_outputs_writes_the_sampled_buffers(tmp_path):
    rng = np.random.default_rng(0)
    n = 300_007
    iv = rng.integers(-2**31, 2**31, n).astype(np.int32)
    dv = rng.integers(-10**7, 10**7, n).astype(np.int64)
    d128 = np.stack([dv, dv >> 63], axis=1)
    d128[5] = (7, 3)                                   # beyond int64: 3 * 2^64 + 7
    xv = rng.standard_normal(n)
    valid = rng.random(n) > 0.1
    bm = _as_u8(np.packbits(valid, bitorder="little"))
    offs = np.concatenate([[0], np.cumsum(rng.integers(0, 44, n))]).astype(np.int32)
    data = rng.integers(0x20, 0x7F, int(offs[-1]) + 32).astype(np.uint8)
    cols = [SimpleNamespace(name=nm, type_id=t) for nm, t in (("i", ch.T_INTEGER), ("d", ch.T_DECIMAL), ("x", ch.T_DOUBLE), ("s", ch.T_VARCHAR))]
    plan = [SimpleNamespace(col=0, op=1, width=4, values=_as_u8(iv), bitmap=bm),
            SimpleNamespace(col=1, op=2, width=16, values=_as_u8(d128), bitmap=bm),
            SimpleNamespace(col=2, op=3, width=8, values=_as_u8(xv), bitmap=bm),
            SimpleNamespace(col=3, op=ch.OP_VALIDITY_ONLY, width=0, values=None, bitmap=bm)]
    step = SimpleNamespace(db=SimpleNamespace(nrows=n, device=torch.device("cpu"), batch=SimpleNamespace(columns=cols)),
                           plan=(plan, None, None), strings=[SimpleNamespace(col=3, mode=0, offsets=_as_u8(offs), data=_as_u8(data))])
    shapes = bench.dump_step_outputs(step, str(tmp_path / "a"))
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")}
    assert set(got) == set(shapes) and all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= bench.DUMP_MAX_BYTES
    rows = got["rows"].astype(np.int64)
    assert rows[0] == 0 and rows[-1] == n - 1 and np.all(np.diff(rows) > 0)
    assert np.array_equal(got["i.values"], iv[rows])
    exp_d = dv[rows].astype(np.float64)
    exp_d[rows == 5] = 3 * 2.0 ** 64 + 7
    assert np.array_equal(got["d.values"], exp_d)
    assert np.array_equal(got["x.values"], xv[rows])
    for c in "idxs":
        assert np.array_equal(got[c + ".validity"], valid[rows])
    assert np.array_equal(got["s.offsets"], np.stack([offs[rows], offs[rows + 1]], axis=1))
    assert np.array_equal(got["s.data"], np.concatenate([data[offs[r]:offs[r + 1]] for r in rows]))
    bench.dump_step_outputs(step, str(tmp_path / "b"))
    for f in os.listdir(tmp_path / "a"):
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
