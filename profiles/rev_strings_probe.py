"""VARCHAR from Arrow string views and dictionaries, against the utf8 path.

Two row shapes, 60 M rows each, 5 % NULL:
  comment    l_comment-like: lengths U[10, 43], so nine rows in ten are pointer string_t
  shipmode   l_shipmode-like: the seven shipping modes, all inline
each as utf8 (rev_string_kernel), utf8_view (rev_view_kernel), dictionary<int8, utf8> over 7 labels and
dictionary<int32, utf8> over 70 000 labels (rev_dict_kernel; a 7-label table sits in shared memory, a 70 000-label one
is read through L2).  Beside them rev_copy (COPY16) of 60 M 16-byte values: the rate a 16 B -> 16 B transform can reach.

Kernel times are CUDA events over `--iters` launches, each case's input in three copies used in turn, so a launch never
finds its input in the 126 MB L2.  Before timing, each encoding's output is checked against the utf8 kernel's on the
same rows: views point into a data buffer laid out as the utf8 one, so every string_t is identical; a dictionary's
pointer string_t point into its own dictionary, so there length and prefix are compared, and inline ones whole.
Algorithmic bytes: what each kernel must read and write (the utf8 kernel: an offset and, per row, the inline bytes or
the 4-byte prefix; views: 16 bytes; indices: their width), plus the bitmap in and the masks out, against the 6454.9
GB/s copy peak DESIGN.md §3 uses.  The whole append (Appender.append_arrow from page-locked host buffers, no sink)
reports the appender's timings and link bytes.

    python profiles/rev_strings_probe.py [--procs 3] [--iters 20] [--out FILE]

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
N = 60_000_000
SHIPMODE = [b"AIR", b"FOB", b"MAIL", b"RAIL", b"REG AIR", b"SHIP", b"TRUCK"]


def _labels(n, rng, lo, hi):
    out, seen = [], set()
    while len(out) < n:
        s = bytes(rng.integers(97, 123, int(rng.integers(lo, hi + 1))).astype(np.uint8))
        if s not in seen:
            seen.add(s)
            out.append(s)
    return out


def _rows(labels, idx):
    """utf8 offsets (int32) and data of labels[idx]"""
    lens = np.asarray([len(x) for x in labels], np.int64)
    off = np.zeros(len(idx) + 1, np.int64)
    np.cumsum(lens[idx], out=off[1:])
    flat = np.frombuffer(b"".join(labels), np.uint8)
    starts = np.concatenate([[0], np.cumsum(lens)])[idx]
    data = np.empty(int(off[-1]) + 64, np.uint8)
    data[-64:] = 0
    for r0 in range(0, len(idx), 1 << 22):  # in blocks: the gather index is 8 bytes per byte
        r1 = min(len(idx), r0 + (1 << 22))
        o0, o1 = int(off[r0]), int(off[r1])
        data[o0:o1] = flat[np.repeat(starts[r0:r1] - off[r0:r1], lens[idx[r0:r1]]) + np.arange(o0, o1)]
    return off.astype(np.int32), data


def _views(off, data, host_base):
    """16-byte views of the utf8 rows (off, data): inline bytes zero-padded, or prefix, buffer 0, the utf8 offset"""
    n = len(off) - 1
    lens = np.diff(off)
    v = np.zeros((n, 16), np.uint8)
    v[:, :4] = lens.astype(np.int32).view(np.uint8).reshape(n, 4)
    for r0 in range(0, n, 1 << 22):
        r1 = min(n, r0 + (1 << 22))
        b12 = data[off[r0:r1, None].astype(np.int64) + np.arange(12)[None, :]]
        ln = lens[r0:r1]
        b12[(np.arange(12)[None, :] >= ln[:, None]) & (ln[:, None] <= 12)] = 0
        ptr = ln > 12
        b12[ptr, 4:8] = 0
        b12[ptr, 8:12] = off[r0:r1][ptr].astype(np.int32).view(np.uint8).reshape(-1, 4)
        v[r0:r1, 4:16] = b12
    return v


def worker(iters: int) -> dict:
    import torch
    sys.path.insert(0, ROOT)
    from duckdb_mbt_b200 import native as nat
    L = nat.lib()
    dev = torch.device("cuda:0")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rng = np.random.default_rng(7)
    res = {"ms": {}, "bytes": {}, "checked": {}}
    HOST = 0x7F0000000000  # the host address the utf8 data buffer and the views' buffer 0 both claim

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

    nch = (N + 2047) // 2048
    outs = {k: torch.empty(nch * 2048 * 16, dtype=torch.uint8, device=dev) for k in ("utf8", "other")}
    val = torch.empty(nch * 32, dtype=torch.int64, device=dev)
    err = torch.full((1,), -1, dtype=torch.int64, device=dev)
    bits = N / 8 + nch * 256

    shapes = {"comment": (lambda n: _labels(n, rng, 10, 43), 10, 43), "shipmode": (lambda n: SHIPMODE if n == 7 else _labels(n, rng, 3, 7), 3, 7)}
    for shape, (make, lo, hi) in shapes.items():
        # the utf8 rows: comment rows all distinct lengths U[10, 43]; shipmode rows the seven modes
        if shape == "comment":
            lens = rng.integers(lo, hi + 1, N)
            off = np.zeros(N + 1, np.int64)
            np.cumsum(lens, out=off[1:])
            data = np.concatenate([rng.integers(32, 127, int(off[-1])).astype(np.uint8), np.zeros(64, np.uint8)])
            off = off.astype(np.int32)
        else:
            off, data = _rows(SHIPMODE, rng.integers(0, 7, N))
        lens = np.diff(off)
        inline = lens <= 12
        bms = [torch.from_numpy(np.packbits(rng.random(N) >= 0.05, bitorder="little")).to(dev) for _ in range(3)]
        d_off = [torch.from_numpy(off).to(dev) for _ in range(3)]
        d_data = [torch.from_numpy(data).to(dev) for _ in range(3)]
        sjobs = [nat.RevStringJob(o.data_ptr(), d.data_ptr(), b.data_ptr(), 0, HOST, outs["utf8"].data_ptr(), val.data_ptr(), None, 0, 0)
                 for o, d, b in zip(d_off, d_data, bms)]
        name = f"{shape}_utf8"
        res["ms"][name] = timed([lambda j=j: nat.check(L.dmb_dev_rev_string_batch(C.byref(j), N, st), name) for j in sjobs])
        res["bytes"][name] = N * 20 + float(np.where(inline, lens, 4).sum()) + bits
        nat.check(L.dmb_dev_rev_string_batch(C.byref(sjobs[0]), N, st), "utf8")
        ref = outs["utf8"].view(-1, 16)[:N].clone()
        torch.cuda.synchronize()
        del sjobs, d_off, d_data
        torch.cuda.empty_cache()
        # views over buffer 0 = the utf8 data buffer at HOST
        views = _views(off, data, HOST)
        d_views = [torch.from_numpy(views).to(dev) for _ in range(3)]
        del views
        table = torch.from_numpy(np.asarray([[HOST, len(data) - 64]], np.int64)).to(dev)
        vjobs = [nat.RevViewJob(v.data_ptr(), b.data_ptr(), 0, table.data_ptr(), 1, outs["other"].data_ptr(), val.data_ptr(), None, err.data_ptr())
                 for v, b in zip(d_views, bms)]
        name = f"{shape}_view"
        nat.check(L.dmb_dev_rev_view_batch(C.byref(vjobs[0]), N, st), name)
        torch.cuda.synchronize()
        res["checked"][name] = bool(torch.equal(outs["other"].view(-1, 16)[:N], ref)) and int(err.item()) == -1
        res["ms"][name] = timed([lambda j=j: nat.check(L.dmb_dev_rev_view_batch(C.byref(j), N, st), name) for j in vjobs])
        res["bytes"][name] = N * 32 + bits
        # COPY16 of the same bytes
        fjobs = [(nat.RevFixedJob * 1)(nat.RevFixedJob(v.data_ptr(), b.data_ptr(), 0, outs["other"].data_ptr(), val.data_ptr(), None, 4, 0))
                 for v, b in zip(d_views, bms)]
        fdev = [torch.from_numpy(np.frombuffer(bytes(f), dtype=np.uint8).copy()).to(dev) for f in fjobs]
        name = f"{shape}_copy16"
        res["ms"][name] = timed([lambda f=f, d=d: nat.check(L.dmb_dev_rev_fixed_batch(d.data_ptr(), C.cast(f, C.c_void_p), 1, N, st), "copy16")
                                 for f, d in zip(fjobs, fdev)])
        res["bytes"][name] = N * 32 + bits
        del d_views, fdev
        torch.cuda.empty_cache()
        # dictionaries: the same row lengths' shape, labels drawn per row
        for dname, nlabels, np_dt, iw in (("dict8", 7, np.int8, 1), ("dict32", 70_000, np.int32, 4)):
            labels = make(nlabels)
            loff, ldata = _rows(labels, np.arange(nlabels))
            lt = torch.from_numpy(ldata).to(dev)
            lo_t = torch.from_numpy(loff).to(dev)
            cap = ((nlabels + 2047) // 2048) * 2048
            tab = torch.zeros(cap * 16, dtype=torch.uint8, device=dev)
            tmask = torch.zeros(cap // 64, dtype=torch.int64, device=dev)
            tj = nat.RevStringJob(lo_t.data_ptr(), lt.data_ptr(), None, 0, HOST, tab.data_ptr(), tmask.data_ptr(), None, 0, 0)
            nat.check(L.dmb_dev_rev_string_batch(C.byref(tj), nlabels, st), "table")
            idxs = [rng.integers(0, nlabels, N).astype(np_dt) for _ in range(3)]
            d_idx = [torch.from_numpy(x).to(dev) for x in idxs]
            djobs = [nat.RevDictJob(x.data_ptr(), b.data_ptr(), 0, tab.data_ptr(), nlabels, outs["other"].data_ptr(), val.data_ptr(), None,
                                    err.data_ptr(), iw, 1) for x, b in zip(d_idx, bms)]
            name = f"{shape}_{dname}"
            # check: the utf8 kernel on the same rows as utf8
            roff, rdata = _rows(labels, idxs[0].astype(np.int64))
            ro, rd = torch.from_numpy(roff).to(dev), torch.from_numpy(rdata).to(dev)
            cj = nat.RevStringJob(ro.data_ptr(), rd.data_ptr(), bms[0].data_ptr(), 0, HOST, outs["utf8"].data_ptr(), val.data_ptr(), None, 0, 0)
            nat.check(L.dmb_dev_rev_string_batch(C.byref(cj), N, st), "utf8 of the dictionary rows")
            nat.check(L.dmb_dev_rev_dict_batch(C.byref(djobs[0]), N, st), name)
            torch.cuda.synchronize()
            g, e = outs["other"].view(-1, 16)[:N], outs["utf8"].view(-1, 16)[:N]
            inl = torch.from_numpy(np.diff(roff) <= 12).to(dev)
            res["checked"][name] = (bool(torch.equal(g[:, :8], e[:, :8])) and bool(torch.equal(g[inl], e[inl])) and int(err.item()) == -1)
            del ro, rd, g, e, inl
            res["ms"][name] = timed([lambda j=j: nat.check(L.dmb_dev_rev_dict_batch(C.byref(j), N, st), name) for j in djobs])
            res["bytes"][name] = N * (iw + 16) + bits + nlabels * 16
            del d_idx
            torch.cuda.empty_cache()
    assert int(err.item()) == -1
    res["share_of_copy_peak"] = {k: res["bytes"][k] / (res["ms"][k] * 1e-3) / 1e9 / PEAK_GBS for k in res["ms"]}
    del outs, val
    torch.cuda.empty_cache()
    res["e2e"] = e2e(rng)
    return res


def e2e(rng) -> dict:
    """the whole append from page-locked host buffers, no sink: each shape as utf8, utf8_view, dictionary<int8, utf8> over 7
    labels and dictionary<int32, utf8> over 70 000 labels of the shape's lengths"""
    import pyarrow as pa
    from duckdb_mbt_b200 import appender as ap
    from duckdb_mbt_b200 import arrow_result as ar
    from duckdb_mbt_b200 import chunks as ch
    from duckdb_mbt_b200 import pinned as pn
    host = []

    def pinned(a):
        p = pn.pinned_empty(a.nbytes)
        p[:] = a.view(np.uint8).reshape(-1)
        host.append(p)
        return pa.foreign_buffer(p.ctypes.data, p.nbytes, base=p)

    out = {}
    valid = pinned(np.packbits(rng.random(N) >= 0.05, bitorder="little"))
    with ar.GpuContext(0) as ctx:
        for shape in ("comment", "shipmode"):
            labels = _labels(7, rng, 10, 43) if shape == "comment" else SHIPMODE
            idx = rng.integers(0, 7, N).astype(np.int8)
            off, data = _rows(labels, idx.astype(np.int64))
            dbuf = pinned(data)
            arrays = {"utf8": pa.Array.from_buffers(pa.string(), N, [valid, pinned(off), dbuf], null_count=-1),
                      "view": pa.Array.from_buffers(pa.string_view(), N, [valid, pinned(_views(off, data, 0)), dbuf], null_count=-1),
                      "dict8": pa.DictionaryArray.from_arrays(pa.Array.from_buffers(pa.int8(), N, [valid, pinned(idx)], null_count=-1),
                                                              pa.array([x.decode() for x in labels])),
                      "dict32": pa.DictionaryArray.from_arrays(
                          pa.Array.from_buffers(pa.int32(), N, [valid, pinned(rng.integers(0, 70_000, N).astype(np.int32))], null_count=-1),
                          pa.array([x.decode() for x in _labels(70_000, rng, *((10, 43) if shape == "comment" else (3, 7)))]))}
            for enc, arr in arrays.items():
                name = f"e2e_{shape}_{enc}"
                out[name] = []
                rb = pa.record_batch([arr], names=["s"])
                for rep in range(6):
                    a = ap.Appender(ctx, [ch.T_VARCHAR], discard=True)
                    a.append_arrow(rb)
                    if rep:  # the first append warms the pools
                        out[name].append(a.timings())
                    a.close()
            del arrays
            host.clear()
            host.append(valid)
    return out


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
        print(json.dumps({"proc": p, "ms": res["ms"], "checked": res["checked"]}), flush=True)
    med = lambda xs: round(statistics.median(xs), 4)  # noqa: E731
    keys = ("h2d_ms", "kernels_ms", "d2h_ms", "total_ms", "h2d_bytes", "d2h_bytes")
    summary = {"card": card, "procs": a.procs, "iters": a.iters, "rows": N,
               "checked_against_utf8": all(all(r["checked"].values()) for r in runs),
               "median_ms": {k: med([r["ms"][k] for r in runs]) for k in runs[0]["ms"]},
               "range_ms": {k: [round(min(r["ms"][k] for r in runs), 4), round(max(r["ms"][k] for r in runs), 4)] for k in runs[0]["ms"]},
               "algorithmic_bytes": runs[0]["bytes"],
               "median_share_of_copy_peak": {k: med([r["share_of_copy_peak"][k] for r in runs]) for k in runs[0]["ms"]},
               "e2e_median": {c: {k: med([x[k] for r in runs for x in r["e2e"][c]]) for k in keys} for c in runs[0]["e2e"]},
               "e2e_total_ms_range": {c: [round(min(x["total_ms"] for r in runs for x in r["e2e"][c]), 3),
                                          round(max(x["total_ms"] for r in runs for x in r["e2e"][c]), 3)] for c in runs[0]["e2e"]}}
    print(json.dumps(summary, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for x in runs:
                f.write(json.dumps(x) + "\n")
            f.write(json.dumps(summary) + "\n")


if __name__ == "__main__":
    main()
