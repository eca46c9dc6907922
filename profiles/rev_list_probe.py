"""The reverse LIST path on 50 M rows of LIST<INTEGER>: Arrow list -> DuckDB LIST vectors.

Lists of U[0, 8] elements (mean 4), 10 % NULL rows, 10 % NULL elements.

  device   L0, device-resident: rev_list_kernel (entries, list masks, per-chunk child masks) plus the child copy
           (rev_fixed_kernel, COPY4) over the whole batch, CUDA events around `--iters` launches of each after a
           warm-up of the same shapes.  Offsets 200 MB and child values 800 MB in, 800 MB of entries and 800 MB of child
           values out: far larger than the 126 MB L2.
  bytes    what the algorithm must move, computed from the shapes: offsets, list bitmap, entries, list masks, child
           values and child bitmap in, child values and child masks out.  Reported against the 6454.9 GB/s copy peak
           DESIGN.md §3 uses.
  e2e      Appender.append_arrow of the same batch from page-locked host buffers (no sink: conversion only), the
           appender's own timings().

    python profiles/rev_list_probe.py [--procs 3] [--iters 20] [--out FILE]

runs one worker process per repetition and prints each worker's numbers and their spread; the card's name and power
limit are read in the same call.
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
N_ROWS = 50_000_000
PEAK_GBS = 6454.9  # DESIGN.md §3: the device-to-device copy peak measured on the B200


def _pack(valid):
    """bool tensor -> LSB-first bitmap bytes (uint8 tensor)"""
    import torch
    pad = (-valid.shape[0]) % 8
    v = torch.cat([valid, torch.zeros(pad, dtype=torch.bool, device=valid.device)]) if pad else valid
    w = torch.tensor([1, 2, 4, 8, 16, 32, 64, 128], dtype=torch.int32, device=valid.device)
    return (v.view(-1, 8).to(torch.int32) * w).sum(1).to(torch.uint8)


def worker(iters: int) -> dict:
    import torch
    sys.path.insert(0, ROOT)
    from duckdb_mbt_b200 import native as nat
    L = nat.lib()
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(3)
    n = N_ROWS
    lens = torch.randint(0, 9, (n,), device=dev, generator=g, dtype=torch.int32)
    off = torch.zeros(n + 1, dtype=torch.int32, device=dev)
    off[1:] = torch.cumsum(lens, 0, dtype=torch.int32)
    e = int(off[-1].item())
    pbm = _pack(torch.rand(n, device=dev, generator=g) >= 0.1)
    child = torch.randint(-2**31, 2**31 - 1, (e,), device=dev, generator=g, dtype=torch.int32)
    cbm = _pack(torch.rand(e, device=dev, generator=g) >= 0.1)
    nch = (n + 2047) // 2048
    idx = torch.clamp(torch.arange(0, nch + 1, device=dev, dtype=torch.int64) * 2048, max=n)
    bnd = off[idx].to(torch.int64)
    cword = torch.zeros(nch + 1, dtype=torch.int64, device=dev)
    cword[1:] = torch.cumsum((bnd[1:] - bnd[:-1] + 63) // 64, 0)
    nwords = int(cword[-1].item())
    ent = torch.empty(nch * 2048 * 16, dtype=torch.uint8, device=dev)
    masks = torch.empty(nch * 32, dtype=torch.int64, device=dev)
    cmasks = torch.empty(nwords + 1, dtype=torch.int64, device=dev)
    cout = torch.empty(e + 16, dtype=torch.int32, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    job = nat.RevListJob(off.data_ptr(), pbm.data_ptr(), 0, cbm.data_ptr(), 0, cword.data_ptr(), ent.data_ptr(), masks.data_ptr(),
                         cmasks.data_ptr(), None, err.data_ptr(), 0, 0)
    fjobs = (nat.RevFixedJob * 1)()
    fjobs[0] = nat.RevFixedJob(child.data_ptr(), cbm.data_ptr(), 0, cout.data_ptr(), None, None, 2, 0)  # DMB_REV_COPY4
    fj_dev = torch.from_numpy(np.frombuffer(bytes(fjobs), dtype=np.uint8).copy()).to(dev)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def run_list():
        nat.check(L.dmb_dev_rev_list_batch(C.byref(job), n, st), "rev_list")

    def run_child():
        nat.check(L.dmb_dev_rev_fixed_batch(fj_dev.data_ptr(), C.cast(fjobs, C.c_void_p), 1, e, st), "rev_fixed")

    def timed(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / iters

    ms_list = timed(run_list)
    ms_child = timed(run_child)
    ms_both = timed(lambda: (run_list(), run_child()))
    assert int(err.item()) == 0
    bytes_list = (n + 1) * 4 + n / 8 + n * 16 + nch * 32 * 8 + e / 8 + nwords * 8
    bytes_child = e * 4 + e / 8 + e * 4
    res = {"rows": n, "elements": e, "ms": {"list_kernel": ms_list, "child_copy": ms_child, "both": ms_both},
           "bytes": {"list_kernel": bytes_list, "child_copy": bytes_child, "both": bytes_list + bytes_child}}
    res["share_of_copy_peak"] = {k: res["bytes"][k] / (res["ms"][k] * 1e-3) / 1e9 / PEAK_GBS for k in res["ms"]}

    # end to end from page-locked host buffers: the appender's own timings
    import pyarrow as pa
    from duckdb_mbt_b200 import appender as ap
    from duckdb_mbt_b200 import arrow_result as ar
    from duckdb_mbt_b200 import chunks as ch
    from duckdb_mbt_b200 import pinned as pn
    host = []

    def pinned(t):
        a = pn.pinned_empty(t.numel() * t.element_size())
        a[:] = t.view(torch.uint8).cpu().numpy()
        host.append(a)
        return pa.foreign_buffer(a.ctypes.data, a.nbytes, base=a)

    child_arr = pa.Array.from_buffers(pa.int32(), e, [pinned(cbm), pinned(child[:e])], null_count=-1)
    arr = pa.Array.from_buffers(pa.list_(pa.int32()), n, [pinned(pbm), pinned(off)], null_count=-1, children=[child_arr])
    rb = pa.record_batch([arr], names=["l"])
    del ent, masks, cmasks, cout
    torch.cuda.empty_cache()
    e2e = []
    with ar.GpuContext(0) as ctx:
        for rep in range(4):
            a = ap.Appender(ctx, [ch.T_LIST], discard=True)
            a.set_list(0, ch.T_INTEGER)
            a.append_arrow(rb)
            if rep:  # the first append warms the pools
                e2e.append(a.timings())
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
        print(json.dumps({"proc": p, "ms": res["ms"], "share_of_copy_peak": res["share_of_copy_peak"],
                          "e2e_total_ms": [round(x["total_ms"], 2) for x in res["e2e"]]}), flush=True)
    med = lambda xs: round(statistics.median(xs), 4)  # noqa: E731
    summary = {"card": card, "rows": N_ROWS, "elements": runs[0]["elements"], "procs": a.procs, "iters": a.iters,
               "median_ms": {k: med([r["ms"][k] for r in runs]) for k in runs[0]["ms"]},
               "range_ms": {k: [round(min(r["ms"][k] for r in runs), 4), round(max(r["ms"][k] for r in runs), 4)] for k in runs[0]["ms"]},
               "algorithmic_bytes": runs[0]["bytes"],
               "median_share_of_copy_peak": {k: med([r["share_of_copy_peak"][k] for r in runs]) for k in runs[0]["ms"]},
               "e2e_median_ms": {k: med([x[k] for r in runs for x in r["e2e"]]) for k in ("h2d_ms", "kernels_ms", "d2h_ms", "total_ms")}}
    print(json.dumps(summary, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for x in runs:
                f.write(json.dumps(x) + "\n")
            f.write(json.dumps(summary) + "\n")


if __name__ == "__main__":
    main()
