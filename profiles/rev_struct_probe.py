"""The reverse STRUCT path: Arrow struct arrays -> DuckDB STRUCT vectors.

  struct_vs_flat  60 M rows of STRUCT{i INTEGER, d DOUBLE, s l_shipmode-like VARCHAR, e uint8 ENUM}, 10 % NULL structs and
                  5 % NULL fields, appended through Appender.append_arrow (no sink), against the same four columns appended
                  flat with the same bitmaps.  Reported: the appender's kernel time (timings()["kernels_ms"], CUDA events
                  around each sub-batch's launches), alternating the two, after one warm-up append of each.
  mask_l0         rev_mask_kernel alone at 60 M rows (two bitmaps at bit offsets 3 and 5 in, one out), CUDA events over
                  `--iters` launches; the inputs are three copies used in turn, so a launch never finds them in L2.
                  Bytes: two bitmaps read, one written.

    python profiles/rev_struct_probe.py [--reps 5] [--iters 50] [--out-dir DIR]

writes one JSON line per case into DIR/rev_struct_probe_b200.jsonl; the card's name and power limit are read in the same
call.
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
SHIPMODE = ["AIR", "FOB", "MAIL", "RAIL", "REG AIR", "SHIP", "TRUCK"]


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--reps", type=int, default=5)
    p.add_argument("--iters", type=int, default=50)
    p.add_argument("--rows", type=int, default=60_000_000)
    p.add_argument("--out-dir", default=None)
    args = p.parse_args()
    import pyarrow as pa
    import torch
    sys.path.insert(0, ROOT)
    from duckdb_mbt_b200 import appender as ap
    from duckdb_mbt_b200 import arrow_result as ar
    from duckdb_mbt_b200 import chunks as ch
    from duckdb_mbt_b200 import native as nat

    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    n = args.rows
    rng = np.random.default_rng(7)
    smask = rng.random(n) < 0.10
    fmask = [rng.random(n) < 0.05 for _ in range(4)]
    e = rng.integers(0, len(SHIPMODE), n).astype(np.uint8)
    labels = pa.array(SHIPMODE)
    fields = [pa.array(rng.integers(-2**31, 2**31 - 1, n).astype(np.int32), mask=fmask[0]),
              pa.array(rng.random(n), mask=fmask[1]),
              pa.DictionaryArray.from_arrays(pa.array(e, mask=fmask[2]), labels).cast(pa.string()),
              pa.DictionaryArray.from_arrays(pa.array(e, mask=fmask[3]), labels)]
    names = ["i", "d", "s", "e"]
    struct_batch = pa.StructArray.from_arrays([pa.StructArray.from_arrays(fields, names=names, mask=pa.array(smask))], names=["st"])
    flat_batch = pa.StructArray.from_arrays(fields, names=names)
    ftypes = [ch.T_INTEGER, ch.T_DOUBLE, ch.T_VARCHAR, ch.T_ENUM]
    lines = []

    with ar.GpuContext(0) as ctx:
        def append(kind):
            if kind == "struct":
                a = ap.Appender(ctx, [ch.T_STRUCT], discard=True)
                first = a.set_struct(0, ftypes)
                a.set_enum(first + 3, SHIPMODE, ch.T_UTINYINT)
                a.append_arrow(struct_batch)
            else:
                a = ap.Appender(ctx, ftypes, discard=True)
                a.set_enum(3, SHIPMODE, ch.T_UTINYINT)
                a.append_arrow(flat_batch)
            t = a.timings()
            a.close()
            return t

        append("struct"), append("flat")  # warm-up: pools, modules
        got = {"struct": [], "flat": []}
        for _ in range(args.reps):
            for kind in ("struct", "flat"):
                got[kind].append(append(kind))
        med = {k: statistics.median(x["kernels_ms"] for x in v) for k, v in got.items()}
        lines.append({"case": "struct_vs_flat", "card": card, "rows": n, "reps": args.reps,
                      "kernels_ms": {k: [round(x["kernels_ms"], 4) for x in v] for k, v in got.items()},
                      "total_ms": {k: [round(x["total_ms"], 3) for x in v] for k, v in got.items()},
                      "median_kernels_ms": {k: round(v, 4) for k, v in med.items()},
                      "struct_over_flat": round(med["struct"] / med["flat"], 4)})
        print(json.dumps(lines[-1]), flush=True)

        # rev_mask_kernel alone
        dev = torch.device("cuda:0")
        nb = (n + 64) // 8 + 16
        ins = [(torch.randint(0, 256, (nb,), dtype=torch.uint8, device=dev), torch.randint(0, 256, (nb,), dtype=torch.uint8, device=dev))
               for _ in range(3)]
        nwords = ((n + 2047) // 2048) * 32
        out = torch.empty(nwords, dtype=torch.int64, device=dev)
        jobs = []
        for a_buf, b_buf in ins:
            j = (nat.RevMaskJob * 1)()
            j[0].in_a, j[0].a_bit_offset, j[0].in_b, j[0].b_bit_offset = a_buf.data_ptr(), 3, b_buf.data_ptr(), 5
            j[0].out, j[0].out_bit_offset = out.data_ptr(), 0
            jobs.append((j, torch.frombuffer(bytearray(bytes(j)), dtype=torch.uint8).to(dev)))
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        L = nat.lib()

        def launch(i):
            j, dj = jobs[i % 3]
            assert L.dmb_dev_rev_mask_batch(dj.data_ptr(), C.addressof(j), 1, n, st) == 0, nat.last_error()

        for i in range(3):
            launch(i)
        torch.cuda.synchronize()
        ms = []
        for _ in range(args.reps):
            s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for i in range(args.iters):
                launch(i)
            t.record()
            torch.cuda.synchronize()
            ms.append(s.elapsed_time(t) / args.iters)
        nbytes = 2 * (n // 8) + nwords * 8
        m = statistics.median(ms)
        lines.append({"case": "mask_l0", "card": card, "rows": n, "iters": args.iters, "ms": [round(x, 4) for x in ms],
                      "median_ms": round(m, 4), "bytes": nbytes, "GB_per_s": round(nbytes / m / 1e6, 1)})
        print(json.dumps(lines[-1]), flush=True)
    if args.out_dir:
        os.makedirs(args.out_dir, exist_ok=True)
        with open(os.path.join(args.out_dir, "rev_struct_probe_b200.jsonl"), "w") as f:
            for x in lines:
                f.write(json.dumps(x) + "\n")


if __name__ == "__main__":
    main()
