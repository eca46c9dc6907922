"""Same-box A/B of the host-API LIST path: duckdb_mb_gpu_result_materialise_arrow on 20 M rows.

Three tables, each with two INTEGER columns beside its LIST column(s):
  flat       LIST<INTEGER> given in dmb_host_list's flat child fields
  described  the same LIST<INTEGER> given as dmb_host_list.child_col
  both       the two LIST columns together
Lists of U[0, 6] elements, 20 % NULL rows, 15 % NULL elements, entries contiguous in row order (what a scan produces),
full 2048-row chunks, every slab in page-locked memory (DMB_BATCH_PINNED).

    python profiles/list_host_ab.py --libs A.so B.so [--passes 5] [--reps 5] [--out FILE]

runs one worker process per (pass, library), the libraries alternating (DMB_LIB_PATH), and prints per library and table
the median of the per-pass medians and their spread (min..max), plus a digest of the exported arrays, so that the
libraries can be checked to compute the same thing.  The card's name and power limit are read in the same call.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_ROWS = 20_000_000


def _build(n, seed=11):
    from duckdb_mbt_b200 import chunks as ch
    from duckdb_mbt_b200 import pinned as pn
    rng = np.random.default_rng(seed)
    V = ch.VECTOR_SIZE
    nch = (n + V - 1) // V
    counts = np.full(nch, V, dtype=np.uint32)
    counts[-1] = n - (nch - 1) * V
    valid = rng.random(n) >= 0.2
    eff = np.where(valid, rng.integers(0, 7, n), 0).astype(np.uint64)
    row_chunk = np.arange(n) // V
    incl = np.cumsum(eff)
    sizes = np.bincount(row_chunk, weights=eff, minlength=nch).astype(np.uint64)
    child_base = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.uint64)
    entries = np.zeros((nch * V, 2), dtype=np.uint64)
    rows = np.arange(n)
    slot = row_chunk * V + rows % V
    entries[slot, 0] = incl - eff - child_base[row_chunk]
    entries[slot, 1] = eff
    entries[slot[~valid]] = rng.integers(1 << 40, 1 << 50, (int((~valid).sum()), 2), dtype=np.uint64)  # never followed
    total = int(sizes.sum())
    child = rng.integers(-2**31, 2**31 - 1, total, dtype=np.int64).astype(np.int32)
    # per-chunk child masks: (size + 63) // 64 + 1 words each, at word offset child_val_off[k]
    words = (sizes + 63) // 64 + 1
    child_val_off = np.concatenate([[0], np.cumsum(words)[:-1]]).astype(np.int64)
    el_chunk = np.repeat(np.arange(nch), sizes.astype(np.int64))
    el_idx = np.arange(total, dtype=np.int64) - child_base[el_chunk].astype(np.int64)
    bits = np.zeros(int(words.sum()) * 64, dtype=np.uint8)
    bits[child_val_off[el_chunk] * 64 + el_idx] = rng.random(total) >= 0.15
    cmask = np.packbits(bits, bitorder="little").view(np.uint64)
    vslab, val_off = ch.make_validity(valid, counts, True)

    entries_p = pn.pinned_copy(entries)
    child_p = pn.pinned_copy(child)
    cmask_p = pn.pinned_copy(cmask).view(np.uint64)
    vslab_p = pn.pinned_copy(vslab).view(np.uint64)
    data_off = np.arange(nch, dtype=np.uint64) * np.uint64(V * 16)

    def flat():
        col = ch.Column("flat", ch.T_LIST, ch.P_U128, entries_p, data_off, vslab_p, val_off)
        col.list_child_type = ch.T_INTEGER
        col.list_child_data, col.list_child_base, col.list_child_sizes = child_p, child_base, sizes
        col.list_child_validity, col.list_child_val_off = cmask_p, child_val_off
        return col

    def described():
        col = ch.Column("described", ch.T_LIST, ch.P_U128, entries_p, data_off, vslab_p, val_off)
        col.list_child_sizes = sizes
        col.list_child_col = ch.Column("item", ch.T_INTEGER, ch.P_I32, child_p, child_base * np.uint64(4), cmask_p, child_val_off)
        return col

    def ints(name, s):
        c = ch.fixed_column(name, ch.T_INTEGER, np.random.default_rng(s).integers(-2**31, 2**31 - 1, n, dtype=np.int64).astype(np.int32),
                            counts, valid=np.random.default_rng(s + 1).random(n) >= 0.1)
        c.data = pn.pinned_copy(c.data)
        c.validity = pn.pinned_copy(c.validity).view(np.uint64)
        return c

    i0, i1 = ints("a", 21), ints("b", 22)
    return {"flat": ch.ChunkBatch(counts, [flat(), i0, i1]),
            "described": ch.ChunkBatch(counts, [described(), i0, i1]),
            "both": ch.ChunkBatch(counts, [flat(), described(), i0, i1])}


def _digest(arr) -> str:
    """offsets, parent and child validity bits, child values: every byte the array defines"""
    h = hashlib.sha256()
    n = len(arr)
    h.update(np.frombuffer(arr.buffers()[1], dtype=np.int32, count=n + 1).tobytes())
    for a in (arr, arr.values):
        bm = a.buffers()[0]
        h.update(np.unpackbits(np.frombuffer(bm, dtype=np.uint8), count=len(a), bitorder="little").tobytes() if bm is not None else b"all")
    h.update(np.frombuffer(arr.values.buffers()[1], dtype=np.int32, count=len(arr.values)).tobytes())
    h.update(arr.type.value_field.name.encode())
    return h.hexdigest()[:16]


def worker(reps: int) -> None:
    sys.path.insert(0, ROOT)
    from duckdb_mbt_b200 import arrow_result as ar
    from duckdb_mbt_b200 import chunks as ch
    batches = _build(N_ROWS)
    out = {"lib": os.environ.get("DMB_LIB_PATH", "default"), "ms": {}, "digest": {}}
    with ar.GpuContext(0) as ctx:
        for name, batch in batches.items():
            times = []
            for rep in range(2 + reps):  # two warm-up passes
                with ar.ArrowResult.from_chunks(ctx, batch, pinned=True) as res:
                    t0 = time.perf_counter()
                    res.materialise()
                    t1 = time.perf_counter()
                    if rep >= 2:
                        times.append((t1 - t0) * 1e3)
                    if rep == 1:
                        out["digest"][name] = [_digest(res.to_arrow(j)) for j in range(len(batch.columns)) if batch.columns[j].type_id == ch.T_LIST]
            out["ms"][name] = times
    print("RESULT " + json.dumps(out), flush=True)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--libs", nargs="+")
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.worker:
        worker(a.reps)
        return
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    runs = []
    for p in range(a.passes):
        order = a.libs if p % 2 == 0 else a.libs[::-1]
        for lib in order:
            env = dict(os.environ, DMB_LIB_PATH=os.path.abspath(lib))
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", "--reps", str(a.reps)], env=env, cwd=ROOT,
                               capture_output=True, text=True)
            line = [x for x in r.stdout.splitlines() if x.startswith("RESULT ")]
            if r.returncode or not line:
                sys.exit(f"worker for {lib} failed ({r.returncode}):\n{r.stdout[-2000:]}\n{r.stderr[-4000:]}")
            res = json.loads(line[0][7:])
            res["pass"] = p
            runs.append(res)
            print(json.dumps({"pass": p, "lib": os.path.basename(lib), "median_ms": {k: round(statistics.median(v), 2) for k, v in res["ms"].items()}}), flush=True)
    summary = {"card": card, "rows": N_ROWS, "passes": a.passes, "reps_per_pass": a.reps, "libs": {}}
    for lib in a.libs:
        mine = [x for x in runs if x["lib"] == os.path.abspath(lib)]
        summary["libs"][os.path.basename(lib)] = {
            name: {"median_ms": round(statistics.median([statistics.median(x["ms"][name]) for x in mine]), 2),
                   "pass_medians_ms": [round(statistics.median(x["ms"][name]), 2) for x in mine],
                   "digest": sorted({"/".join(x["digest"][name]) for x in mine})}
            for name in mine[0]["ms"]}
    print(json.dumps(summary, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for x in runs:
                f.write(json.dumps(x) + "\n")
            f.write(json.dumps(summary) + "\n")


if __name__ == "__main__":
    main()
