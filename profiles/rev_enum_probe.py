"""The reverse ENUM path: Arrow dictionary indices and utf8 labels -> DuckDB ENUM positions.

  idx_u8      60 M uint8 dictionary indices, 7 labels -> uint8 ENUM (remap in shared memory); beside it rev_copy (COPY1) of the
              same bytes, which is what an identity special case could at best cost
  idx_i32     60 M int32 indices into a 70 000-label dictionary -> uint32 ENUM (remap read through L2)
  str_short   60 M utf8 rows drawn from 7 short labels (l_shipmode-like) -> uint8 ENUM (table in shared memory)
  str_10k     30 M utf8 rows drawn from 10 000 labels of 8-24 bytes -> uint16 ENUM (table read through L2)
  e2e         Appender.append_arrow of the idx_u8 and str_short batches from page-locked host buffers (no sink), the
              appender's own timings()

Every input is 5 % NULL.  Each case is warmed up, then timed with CUDA events over `--iters` launches; the inputs of each
case are three copies used in turn, so a launch never finds its input in the 126 MB L2.  Algorithmic bytes: indices (or
offsets + label bytes) and the bitmap in, the remap table once, positions and masks out; against the 6454.9 GB/s copy
peak DESIGN.md §3 uses.

    python profiles/rev_enum_probe.py [--procs 3] [--iters 20] [--out FILE]

runs one worker process per repetition; the card's name and power limit are read in the same call.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PEAK_GBS = 6454.9
SHIPMODE = [b"AIR", b"FOB", b"MAIL", b"RAIL", b"REG AIR", b"SHIP", b"TRUCK"]


def _labels(n, rng, lo, hi):
    out, seen = [], set()
    while len(out) < n:
        s = bytes(rng.integers(97, 123, int(rng.integers(lo, hi + 1))).astype(np.uint8))
        if s not in seen:
            seen.add(s)
            out.append(s)
    return out


def worker(iters: int) -> dict:
    import torch
    sys.path.insert(0, ROOT)
    from duckdb_mbt_b200 import appender as ap
    from duckdb_mbt_b200 import native as nat
    L = nat.lib()
    dev = torch.device("cuda:0")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rng = np.random.default_rng(5)
    res = {"ms": {}, "bytes": {}}

    def timed(fns):
        for fn in fns:
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(iters):
            fns[i % len(fns)]()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / iters

    def bitmap(n):
        return torch.from_numpy(np.packbits(rng.random(n) >= 0.05, bitorder="little")).to(dev)

    def out_bufs(n, w):
        nch = (n + 2047) // 2048
        return torch.empty(nch * 2048 * w, dtype=torch.uint8, device=dev), torch.empty(nch * 32, dtype=torch.int64, device=dev)

    err = torch.full((1,), -1, dtype=torch.int64, device=dev)

    def table_of(labels):
        d, keep = ap.enum_dict(labels)
        size = 16
        while size < 2 * len(labels):
            size *= 2
        slots = np.zeros(size * 32, np.uint8)
        assert L.dmb_rev_enum_table(C.byref(d), size, slots.ctypes.data)
        offs, data = keep
        return (torch.from_numpy(slots).to(dev), size, torch.from_numpy(offs.view(np.uint8).copy()).to(dev),
                torch.from_numpy(np.concatenate([data, np.zeros(64, np.uint8)])).to(dev))

    # ---- dictionary indices
    def idx_case(name, n, nlabels, np_dt, iw, ow):
        remap = torch.from_numpy(rng.permutation(nlabels).astype(np.uint32)).to(dev)
        ins = [torch.from_numpy(rng.integers(0, nlabels, n).astype(np_dt)).to(dev) for _ in range(3)]
        bms = [bitmap(n) for _ in range(3)]
        out, val = out_bufs(n, ow)
        jobs = [nat.RevEnumJob(in_indices=x.data_ptr(), in_validity=b.data_ptr(), remap=remap.data_ptr(), dict_len=nlabels,
                               out=out.data_ptr(), out_validity=val.data_ptr(), error=err.data_ptr(), out_width=ow, index_width=iw)
                for x, b in zip(ins, bms)]
        res["ms"][name] = timed([lambda j=j: nat.check(L.dmb_dev_rev_enum_batch(C.byref(j), n, st), name) for j in jobs])
        res["bytes"][name] = n * (iw + ow) + n / 8 + ((n + 2047) // 2048) * 256 + nlabels * 4
        return ins, bms, out

    ins, bms, out = idx_case("idx_u8", 60_000_000, 7, np.uint8, 1, 1)
    n = 60_000_000
    fjobs = [(nat.RevFixedJob * 1)(nat.RevFixedJob(x.data_ptr(), b.data_ptr(), 0, out.data_ptr(), None, None, 0, 0)) for x, b in zip(ins, bms)]
    fdev = [torch.from_numpy(np.frombuffer(bytes(f), dtype=np.uint8).copy()).to(dev) for f in fjobs]
    res["ms"]["rev_copy_u8"] = timed([lambda f=f, d=d: nat.check(L.dmb_dev_rev_fixed_batch(d.data_ptr(), C.cast(f, C.c_void_p), 1, n, st), "copy")
                                      for f, d in zip(fjobs, fdev)])
    res["bytes"]["rev_copy_u8"] = 2 * n + n / 8
    del ins, bms, out
    idx_case("idx_i32", 60_000_000, 70_000, np.int32, 4, 4)
    torch.cuda.empty_cache()

    # ---- utf8 labels
    def str_case(name, n, labels, ow):
        tab, size, loff, ldata = table_of(labels)
        lens = np.asarray([len(x) for x in labels])
        jobs, keep = [], []
        out, val = out_bufs(n, ow)
        for _ in range(3):
            pick = rng.integers(0, len(labels), n)
            off = np.zeros(n + 1, np.int64)
            np.cumsum(lens[pick], out=off[1:])
            flat = np.frombuffer(b"".join(labels), np.uint8)
            starts = np.concatenate([[0], np.cumsum(lens)])[pick]
            gather = np.repeat(starts - off[:-1], lens[pick]) + np.arange(off[-1])
            data = torch.from_numpy(np.concatenate([flat[gather], np.zeros(64, np.uint8)])).to(dev)
            o = torch.from_numpy(off.astype(np.int32)).to(dev)
            b = bitmap(n)
            keep += [data, o, b]
            jobs.append(nat.RevEnumJob(in_offsets=o.data_ptr(), in_data=data.data_ptr(), in_validity=b.data_ptr(), table=tab.data_ptr(),
                                       label_offsets=loff.data_ptr(), label_data=ldata.data_ptr(), out=out.data_ptr(), out_validity=val.data_ptr(),
                                       error=err.data_ptr(), table_size=size, out_width=ow))
            mean_len = float(lens[pick].mean())
        res["ms"][name] = timed([lambda j=j: nat.check(L.dmb_dev_rev_enum_batch(C.byref(j), n, st), name) for j in jobs])
        res["bytes"][name] = n * (4 + mean_len + ow) + n / 8 + ((n + 2047) // 2048) * 256
        return keep

    str_case("str_short", 60_000_000, SHIPMODE, 1)
    torch.cuda.empty_cache()
    str_case("str_10k", 30_000_000, _labels(10_000, rng, 8, 24), 2)
    torch.cuda.empty_cache()
    assert int(err.item()) == -1
    res["share_of_copy_peak"] = {k: res["bytes"][k] / (res["ms"][k] * 1e-3) / 1e9 / PEAK_GBS for k in res["ms"]}

    # ---- end to end from page-locked host buffers
    import pyarrow as pa
    from duckdb_mbt_b200 import arrow_result as ar
    from duckdb_mbt_b200 import chunks as ch
    from duckdb_mbt_b200 import pinned as pn
    n = 60_000_000
    host = []

    def pinned(a):
        p = pn.pinned_empty(a.nbytes)
        p[:] = a.view(np.uint8).reshape(-1)
        host.append(p)
        return pa.foreign_buffer(p.ctypes.data, p.nbytes, base=p)

    valid = np.packbits(rng.random(n) >= 0.05, bitorder="little")
    idx = rng.integers(0, 7, n).astype(np.uint8)
    dict_arr = pa.DictionaryArray.from_arrays(pa.Array.from_buffers(pa.uint8(), n, [pinned(valid), pinned(idx)], null_count=-1),
                                              pa.array([x.decode() for x in SHIPMODE]))
    lens = np.asarray([len(x) for x in SHIPMODE])
    off = np.zeros(n + 1, np.int32)
    np.cumsum(lens[idx], out=off[1:])
    str_arr = dict_arr.dictionary.take(pa.array(idx)).cast(pa.string())
    str_arr = pa.Array.from_buffers(pa.string(), n, [pinned(valid), pinned(off), pinned(np.frombuffer(str_arr.buffers()[2], np.uint8)[: off[-1]].copy())],
                                    null_count=-1)
    e2e = {}
    with ar.GpuContext(0) as ctx:
        for name, arr in (("e2e_idx_u8", dict_arr), ("e2e_str_short", str_arr)):
            rb = pa.record_batch([arr], names=["e"])
            e2e[name] = []
            for rep in range(4):
                a = ap.Appender(ctx, [ch.T_ENUM], discard=True)
                a.set_enum(0, SHIPMODE, ch.T_UTINYINT)
                a.append_arrow(rb)
                if rep:  # the first append warms the pools
                    e2e[name].append(a.timings())
                a.close()
    res["e2e"] = e2e
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--procs", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.worker:
        print("RESULT " + json.dumps(worker(a.iters)), flush=True)
        return
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    runs = []
    for p in range(a.procs):
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", "--iters", str(a.iters)], cwd=ROOT,
                           capture_output=True, text=True)
        line = [x for x in r.stdout.splitlines() if x.startswith("RESULT ")]
        if r.returncode or not line:
            sys.exit(f"worker failed ({r.returncode}):\n{r.stdout[-2000:]}\n{r.stderr[-4000:]}")
        res = json.loads(line[0][7:])
        res["proc"] = p
        runs.append(res)
        print(json.dumps({"proc": p, "ms": res["ms"], "share_of_copy_peak": res["share_of_copy_peak"]}), flush=True)
    med = lambda xs: round(statistics.median(xs), 4)  # noqa: E731
    summary = {"card": card, "procs": a.procs, "iters": a.iters,
               "median_ms": {k: med([r["ms"][k] for r in runs]) for k in runs[0]["ms"]},
               "range_ms": {k: [round(min(r["ms"][k] for r in runs), 4), round(max(r["ms"][k] for r in runs), 4)] for k in runs[0]["ms"]},
               "algorithmic_bytes": runs[0]["bytes"],
               "median_share_of_copy_peak": {k: med([r["share_of_copy_peak"][k] for r in runs]) for k in runs[0]["ms"]},
               "e2e_median_ms": {c: {k: med([x[k] for r in runs for x in r["e2e"][c]]) for k in ("h2d_ms", "kernels_ms", "d2h_ms", "total_ms")}
                                 for c in runs[0]["e2e"]}}
    print(json.dumps(summary, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for x in runs:
                f.write(json.dumps(x) + "\n")
            f.write(json.dumps(summary) + "\n")


if __name__ == "__main__":
    main()
