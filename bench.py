#!/usr/bin/env python
"""bench.py — DataChunk -> Arrow materialisation throughput (BASELINE.json metric) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--rows R] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload of `value` (config.workload): BASELINE.json configs[1], the synthetic lineitem-shaped table
(4 INTEGER, 4 DECIMAL(15,2), 3 DATE, 5 VARCHAR; 60 M rows per GPU, no NULLs) -> Arrow record batch.
One step = one pass of the hot path over the whole table.  Row groups shard across GPUs with no
data-path collective (SURVEY.md §8e): every rank converts its own 60 M-row range of the table, scaling
"weak"; torch.distributed (NCCL) is used for the barrier, the max-over-ranks timing and the gather of
the per-GPU string byte totals (the host exclusive scan that rebases offsets across GPUs).

  value        rows/s, inputs resident in HBM, CUDA events on the launching stream, max over ranks
  parity       BEFORE anything is timed, sampled chunk windows of every output column of every config
               are compared bit for bit with the CPU oracle (parity_checked_rows)
  e2e          rows/s through the reference-facing C ABI (duckdb_mb_gpu_result_from_chunks +
               _materialise_arrow) with page-locked HOST buffers, H2D + kernels + D2H in the timed region
  e2e_duckdb_layout   the same call on the input the glue really hands over: one pageable buffer per
               2048-row vector, flags = 0, scattered per-chunk string heaps (heap_len = 0), no hints
  e2e_getters  the reference's own surface: 16 duckdb_mb_arrow_get_column_*_nullable calls + the decoder
               mirror per 1 M-row result (what --impl reference times on the CPU)
  configs      C1 / C3 / C4 / C5 of BASELINE.json, device-resident, in the same clock-sampled region; LIST / ENUM
               (SURVEY.md 8f item 3: LIST<INTEGER> -> Arrow list<int32>, ENUM -> utf8) at the device API beside them
  roofline     the dominant kernel family of the C2 step: algorithmic bytes / its CUDA-event time
  cpu_baseline the oracle port of the reference's getters + decoders, 1 core, <= 1 M-row sample;
  cpu_columnar an -O3 -march=native OpenMP columnar conversion on all host cores (oracle/columnar.c)

`--dump-outputs DIR` writes, after the timed steps, what the last timed step of `value` computed on rank 0 (a fixed, seeded
sample of its rows; see dump_step_outputs) as DIR/<name>.npy, so that two builds can be compared output for output.

`--impl reference` times the reference's own CPU path (oracle port: the reference cannot be built
here, SURVEY.md §8c) on the host cores.  Nothing here reads /root/reference.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "datachunk_to_arrow_rows_per_s"
UNIT = "rows/s"
DEFAULT_ROWS = 60_000_000
CPU_SAMPLE_ROWS = 1_000_000  # the reference's decoders return [] above this (src/duckdb_arrow_native.mbt:435)
WINDOW_CHUNKS = 489          # parity windows: ~1 M rows of whole chunks
GETTER_CHUNKS = 488          # e2e_getters results: 999 424 rows, just under the reference decoders' 1 000 000-row cap
VS = 2048
DUMP_ROWS = 1 << 16          # --dump-outputs: sampled rows of the C2 step (~28 MB of .npy at the default table)
DUMP_MAX_BYTES = 64 << 20


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md)."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa_node(index: int) -> None:
    """Run this rank (and first-touch its page-locked buffers) on the CPUs next to its GPU."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        allowed = os.sched_getaffinity(0)
        if cpus & allowed:
            os.sched_setaffinity(0, cpus & allowed)
    except Exception:
        pass


def mem_available_gb() -> float:
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable"):
                return int(ln.split()[1]) / 1e6
    except OSError:
        pass
    return 1e9


def measure_host_link(device, barrier, nbytes=1 << 30, iters=3):
    """Pinned cudaMemcpyAsync bandwidth of this GPU's host link (GB/s): H2D alone, D2H alone, both at once.  Every
    measurement starts behind a barrier, so at N GPUs the figures are what the links give when ALL ranks copy at
    the same time (the ceiling the e2e legs are judged against, BASELINE.json metric: % of host-link)."""
    import torch
    h_in = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    h_out = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d_a = torch.empty(nbytes, dtype=torch.uint8, device=device)
    d_b = torch.empty(nbytes, dtype=torch.uint8, device=device)
    s1, s2 = torch.cuda.Stream(device), torch.cuda.Stream(device)

    def run(h2d, d2h):
        barrier()
        t0 = time.perf_counter()
        for _ in range(iters):
            if h2d:
                with torch.cuda.stream(s1):
                    d_a.copy_(h_in, non_blocking=True)
            if d2h:
                with torch.cuda.stream(s2):
                    h_out.copy_(d_b, non_blocking=True)
        torch.cuda.synchronize(device)
        return iters * nbytes / (time.perf_counter() - t0) / 1e9

    run(True, True)
    out = {"h2d_gbs": run(True, False), "d2h_gbs": run(False, True)}
    both = run(True, True)
    out["bidir_each_gbs"] = both
    out["bidir_sum_gbs"] = 2 * both
    out["concurrent_ranks"] = True
    del h_in, h_out, d_a, d_b
    return out


# ----------------------------------------------------------------------------- workloads
def build_c2_device(nrows: int, seed: int, device, host_heap_alloc=None):
    """BASELINE.json configs[1] generated directly in HBM (SURVEY.md §8d C2)."""
    import torch
    from duckdb_mbt_b200 import chunks as ch
    from duckdb_mbt_b200 import devgen

    gen = torch.Generator(device=device)
    gen.manual_seed(seed)
    b = devgen.GeneratedBatch(nrows, device)
    for nm in ("l_orderkey", "l_partkey", "l_suppkey", "l_linenumber"):
        b.add_fixed(ch.T_INTEGER, 0, gen, 0.0, nm, lo=0, hi=2**31 - 1)
    for nm in ("l_quantity", "l_extendedprice", "l_discount", "l_tax"):
        b.add_fixed(ch.T_DECIMAL, 15, gen, 0.0, nm, lo=0, hi=10**7, dec_scale=2)
    for nm in ("l_shipdate", "l_commitdate", "l_receiptdate"):
        b.add_fixed(ch.T_DATE, 0, gen, 0.0, nm, lo=8035, hi=10592)
    kw = dict(host_heap_alloc=host_heap_alloc)
    b.add_string(gen, 0.0, 1, 1, name="l_returnflag", **kw)
    b.add_string(gen, 0.0, 1, 1, name="l_linestatus", **kw)
    b.add_string(gen, 0.0, 0, 0, name="l_shipinstruct", len_choices=[17, 11, 4, 16], **kw)
    b.add_string(gen, 0.0, 0, 0, name="l_shipmode", len_choices=[7, 3, 4, 4, 5, 4, 3], **kw)
    b.add_string(gen, 0.0, 10, 43, name="l_comment", **kw)
    return b


def arrow_dst(col):
    from duckdb_mbt_b200 import chunks as ch
    return ch.D_I128 if col.type_id in (ch.T_DECIMAL, ch.T_HUGEINT) else ch.D_SAME


class DeviceStep:
    """One pass of the hot path with inputs resident in HBM (device API, L0): every fixed-width column in one launch per
    distinct conversion, every VARCHAR column in one launch.  `large`: int64 utf8 offsets (C3: > 2^31 string bytes)."""

    def __init__(self, db, large=False):
        import torch
        from duckdb_mbt_b200 import chunks as ch
        self.torch = torch
        self.db = db
        cols = db.batch.columns
        fixed = [j for j, c in enumerate(cols) if c.phys != ch.P_STRING]
        strings = [j for j, c in enumerate(cols) if c.phys == ch.P_STRING]
        specs = [(j, arrow_dst(cols[j])) for j in fixed] + [(j, ch.OP_VALIDITY_ONLY) for j in strings]
        self.plan = db.plan_fixed(specs, bitmap=True)
        self.mode = 1 if large else 0
        self.strings = [db.plan_string(j, self.mode, data_capacity=db.meta[j]["total_len"]) for j in strings]
        n = db.nrows
        self.alg_fixed = db.alg_bytes_fixed(self.plan)
        ow = 8 if large else 4
        self.alg_string = sum(16 * n + db.meta[j]["ptr_len"] + ow * (n + 1) + db.meta[j]["total_len"] for j in strings)
        self.n_fixed_launches = len({o.op for o in self.plan[0]})
        self.launches = self.n_fixed_launches + len(self.strings)

    def run(self, record=False):
        torch = self.torch
        if record:
            e0, e1 = (torch.cuda.Event(enable_timing=True) for _ in range(2))
            e0.record()
        self.db.run_fixed(self.plan)
        if record:
            e1.record()
        marks = []
        for so in self.strings:
            self.db.run_string(so)
            if record:
                m = torch.cuda.Event(enable_timing=True)
                m.record()
                marks.append(m)
        if record:
            return e0, e1, (marks[-1] if marks else e1), marks
        return None

    def check(self):
        for so in self.strings:
            if self.db.string_error(so) != 0:
                from duckdb_mbt_b200 import native as nat
                raise RuntimeError("string kernel flagged an error: " + nat.last_error())


def dump_step_outputs(step: DeviceStep, out_dir: str, seed: int = 0) -> dict:
    """Write the Arrow buffers a DeviceStep's last run produced, at a fixed, seeded sample of DUMP_ROWS rows (always the
    first and the last), as out_dir/<name>.npy:
      rows.npy                  the sampled row indices (float64, ascending)
      <column>.values.npy       fixed-width values (float64; decimal128 / hugeint as the unscaled integer, exact up to 2^53)
      <column>.validity.npy     the validity bit of every sampled row (float32 0 / 1), every column
      <column>.offsets.npy      utf8 offsets (start, end) of every sampled row (float64, shape (rows, 2))
      <column>.data.npy         the sampled rows' utf8 bytes, concatenated in row order (float32)
    The sample depends only on the row count and the seed, so runs with the same arguments write comparable files.
    Returns {file name: shape}."""
    import numpy as np
    import torch
    from duckdb_mbt_b200 import chunks as ch
    db = step.db
    n = db.nrows
    rng = np.random.default_rng(seed)
    rows = np.unique(np.concatenate([[0, n - 1], rng.integers(0, n, max(DUMP_ROWS - 2, 0))]))
    idx = torch.from_numpy(rows).to(db.device)
    out = {"rows": rows.astype(np.float64)}
    for o in step.plan[0]:
        name = db.batch.columns[o.col].name
        bits = o.bitmap[: (n + 7) // 8][idx // 8].to(torch.int32) >> (idx % 8).to(torch.int32)
        out[name + ".validity"] = (bits & 1).cpu().numpy().astype(np.float32)
        if o.op == ch.OP_VALIDITY_ONLY:
            continue
        w = o.width
        v = o.values[: n * w].view(n, w)[idx].cpu().numpy()
        if w == 16:
            lo, hi = v.view(np.int64)[:, 0], v.view(np.int64)[:, 1]
            out[name + ".values"] = np.where(hi == lo >> 63, lo.astype(np.float64),
                                             hi.astype(np.float64) * 2.0 ** 64 + lo.view(np.uint64).astype(np.float64))
        else:
            float_type = {4: ch.T_FLOAT, 8: ch.T_DOUBLE}.get(w)
            dt = np.dtype(("f" if db.batch.columns[o.col].type_id == float_type else "i") + str(w))
            out[name + ".values"] = v.view(dt).reshape(-1).astype(np.float64)
    for so in step.strings:
        name = db.batch.columns[so.col].name
        offs = so.offsets[: (n + 1) * (8 if so.mode == 1 else 4)].view(torch.int64 if so.mode == 1 else torch.int32)
        start, end = offs[idx].to(torch.int64), offs[idx + 1].to(torch.int64)
        lens = end - start
        first = torch.cumsum(lens, 0) - lens
        pos = torch.repeat_interleave(start - first, lens) + torch.arange(int(lens.sum().item()), device=db.device)
        out[name + ".offsets"] = torch.stack([start, end], dim=1).cpu().numpy().astype(np.float64)
        out[name + ".data"] = so.data[pos].cpu().numpy().astype(np.float32)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte cap")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return {name: list(a.shape) for name, a in out.items()}


# ----------------------------------------------------------------------------- parity before timing (oracle = checker)
def windows(nchunks: int, seed: int, k: int = 1, size: int = WINDOW_CHUNKS):
    """chunk ranges [c0, c1): the head, the tail (ragged last chunk) and k seeded random ones"""
    import numpy as np
    size = min(size, nchunks)
    out = [(0, size), (nchunks - size, nchunks)]
    rng = np.random.default_rng(seed)
    for _ in range(k):
        c0 = int(rng.integers(0, nchunks - size + 1))
        out.append((c0, c0 + size))
    return out


def parity_check_step(step: DeviceStep, seed: int, k: int = 1) -> int:
    """Compare sampled chunk windows of EVERY output column of a DeviceStep with the CPU oracle, bit for bit.  The device
    converted the whole column; the oracle converts the window's chunks (devgen.window_to_host) and the window is cut out
    of the device output (utf8 offsets rebased by the window's first offset).  Returns the number of cells compared;
    raises AssertionError on the first difference."""
    import numpy as np
    import oracle
    from duckdb_mbt_b200 import chunks as ch
    db = step.db
    checked = 0
    for c0, c1 in windows(db.nchunks, seed, k):
        sub = db.window_to_host(c0, c1)
        ora = oracle.OracleResult(sub)
        row0, nw = c0 * VS, sub.nrows
        nb = (nw + 7) // 8
        tail = nw % 8

        def bitmap_equal(dev_bitmap, exp):
            got = dev_bitmap[row0 // 8: row0 // 8 + nb].cpu().numpy().copy()
            exp = exp[:nb].copy()
            if tail:
                got[-1] &= (1 << tail) - 1
                exp[-1] &= (1 << tail) - 1
            return np.array_equal(got, exp)

        for o in step.plan[0]:
            if o.op == ch.OP_VALIDITY_ONLY:
                _, bm, _, _ = ora.arrow_fixed(o.col, ch.D_SAME, 16, want_values=False)
            else:
                ev, bm, _, _ = ora.arrow_fixed(o.col, o.op & 0xFF, o.width)
                got = o.values[row0 * o.width: row0 * o.width + ev.shape[0]].cpu().numpy()
                assert np.array_equal(got, ev), f"parity: values of column {o.col} differ from the oracle (chunks {c0}..{c1})"
            assert bitmap_equal(o.bitmap, bm), f"parity: validity bitmap of column {o.col} differs (chunks {c0}..{c1})"
            checked += nw
        for so in step.strings:
            ow = 8 if so.mode == 1 else 4
            offs = so.offsets[row0 * ow: (row0 + nw + 1) * ow].cpu().numpy().view(np.int64 if so.mode == 1 else np.int32).astype(np.int64)
            eo, ed = ora.arrow_string(so.col, 1)
            base = int(offs[0])
            assert np.array_equal(offs - base, eo), f"parity: utf8 offsets of column {so.col} differ (chunks {c0}..{c1})"
            got = so.data[base: base + ed.shape[0]].cpu().numpy()
            assert np.array_equal(got, ed), f"parity: utf8 data of column {so.col} differs (chunks {c0}..{c1})"
        ora.close()
    return checked


class ReverseStep:
    """BASELINE.json configs[4] (C5), one device-resident batch: Arrow int32 id, int64 v, float64 x, bool flag, utf8 s
    (len U[0,24]); 10 % NULL except id; every column a slice at a non-zero element / bit offset -> DataChunk vectors."""
    OFF = 3

    def __init__(self, n, seed, device):
        import numpy as np
        import torch
        from duckdb_mbt_b200 import native as nat
        self.torch, self.nat, self.n, self.device = torch, nat, n, device
        L = self.L = nat.lib()
        off = self.OFF
        gen = torch.Generator(device=device)
        gen.manual_seed(seed)
        nch = (n + VS - 1) // VS

        def bitmap(frac):
            m = (n + off + 64) // 8 * 8
            bits = torch.rand(m, generator=gen, device=device) >= frac
            w = torch.tensor([1, 2, 4, 8, 16, 32, 64, 128], dtype=torch.int32, device=device)
            return (bits.view(-1, 8).to(torch.int32) * w).sum(dim=1).to(torch.uint8)

        self.ids = torch.arange(n + off, dtype=torch.int32, device=device)
        self.v = torch.randint(-2**62, 2**62, (n + off,), generator=gen, device=device, dtype=torch.int64)
        self.x = torch.rand(n + off, generator=gen, device=device, dtype=torch.float64)
        self.flag = bitmap(0.5)
        self.masks = [None, bitmap(0.1), bitmap(0.1), bitmap(0.1), bitmap(0.1)]
        lens = torch.randint(0, 25, (n + off,), generator=gen, device=device, dtype=torch.int64)
        offs64 = torch.zeros(n + off + 1, dtype=torch.int64, device=device)
        torch.cumsum(lens, 0, out=offs64[1:])
        total = int(offs64[-1].item())
        self.live = int((offs64[n + off] - offs64[off]).item())
        self.offs = offs64.to(torch.int32)
        del offs64, lens
        self.data = torch.randint(0x20, 0x7F, (total + 64,), generator=gen, device=device, dtype=torch.uint8)
        self.widths = [4, 8, 8, 1, 16]
        self.outs = [torch.empty(nch * VS * w + 64, dtype=torch.uint8, device=device) for w in self.widths]
        self.vals = [torch.empty(nch * 32 * 8 + 64, dtype=torch.uint8, device=device) for _ in range(5)]
        self.data_host_base = 0x7F0000000000
        jobs = (nat.RevFixedJob * 4)()
        jobs[0] = nat.RevFixedJob(self.ids.data_ptr() + 4 * off, None, off, self.outs[0].data_ptr(), self.vals[0].data_ptr(), None, 2, 0)
        jobs[1] = nat.RevFixedJob(self.v.data_ptr() + 8 * off, self.masks[1].data_ptr(), off, self.outs[1].data_ptr(), self.vals[1].data_ptr(), None, 3, 0)
        jobs[2] = nat.RevFixedJob(self.x.data_ptr() + 8 * off, self.masks[2].data_ptr(), off, self.outs[2].data_ptr(), self.vals[2].data_ptr(), None, 3, 0)
        jobs[3] = nat.RevFixedJob(self.flag.data_ptr(), self.masks[3].data_ptr(), off, self.outs[3].data_ptr(), self.vals[3].data_ptr(), None, 5, 0)
        self.jobs = jobs
        self.jobs_dev = torch.from_numpy(np.frombuffer(bytes(jobs), dtype=np.uint8).copy()).to(device)
        self.sjob = nat.RevStringJob(self.offs.data_ptr() + 4 * off, self.data.data_ptr(), self.masks[4].data_ptr(), off, self.data_host_base,
                                     self.outs[4].data_ptr(), self.vals[4].data_ptr(), None, 0, 0)
        # SURVEY.md §8d reverse accounting: Arrow buffers read once, vectors + masks written; string bytes are read for
        # the prefix / inline fill only (pointer strings refer to the Arrow data buffer in place)
        self.alg_string = 4 * (n + 1) + self.live + 16 * n + 2 * (n // 8)
        self.alg_fixed = n * (4 + 4) + n * (8 + 8) * 2 + (n // 8 + n) + 4 * (n // 8) * 2 + n // 8
        self.launches = 5  # rev_fixed_kernel: one launch per job (grid.y), reported as launches of the family

    def run(self, record=False):
        torch, nat, L = self.torch, self.nat, self.L
        stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        if record:
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            e0.record()
        nat.check(L.dmb_dev_rev_fixed_batch(self.jobs_dev.data_ptr(), C.cast(self.jobs, C.c_void_p), 4, self.n, stream), "rev_fixed")
        if record:
            e1.record()
        nat.check(L.dmb_dev_rev_string_batch(C.byref(self.sjob), self.n, stream), "rev_string")
        if record:
            e2.record()
            return e0, e1, e2
        return None

    def parity_check(self, seed: int) -> int:
        """windows of whole 2048-row chunks of every output slab against the oracle's reverse restatement"""
        import numpy as np
        import oracle
        n, off = self.n, self.OFF
        nch = (n + VS - 1) // VS
        checked = 0
        for c0, c1 in windows(nch, seed, 1):
            r0, r1 = c0 * VS, min(c1 * VS, n)
            nw = r1 - r0
            srcs = [(self.ids, 4, 2), (self.v, 8, 3), (self.x, 8, 3)]
            for j, (t, w, op) in enumerate(srcs):
                vals = t.view(torch_uint8())[(off + r0) * w: (off + r1) * w].cpu().numpy()
                bm, boff = self._bitmap_window(j, r0, nw)
                exp_out, exp_val, _ = oracle.rev_fixed(vals, bm, boff, nw, op, w)
                self._cmp(j, c0, r0, nw, w, exp_out, exp_val)
            p = off + r0
            bits = self.flag[p // 8: (p + nw + 7) // 8 + 1].cpu().numpy()
            bm, boff = self._bitmap_window(3, r0, nw)
            # value bits and validity bits start at the same bit offset (same array offset)
            exp_out, exp_val, _ = oracle.rev_fixed(bits, bm, boff, nw, 5, 1)
            self._cmp(3, c0, r0, nw, 1, exp_out, exp_val)
            offs = self.offs[off + r0: off + r1 + 1].cpu().numpy()
            o0, o1 = int(offs[0]), int(offs[-1])
            data = self.data[o0: o1 + 16].cpu().numpy()
            bm, boff = self._bitmap_window(4, r0, nw)
            exp_out, exp_val, _ = oracle.rev_string(np.ascontiguousarray(offs - o0), data, self.data_host_base + o0, bm, boff, nw)
            self._cmp(4, c0, r0, nw, 16, exp_out, exp_val)
            checked += 5 * nw
        return checked

    def _bitmap_window(self, j, r0, nw):
        m = self.masks[j]
        if m is None:
            return None, 0
        p = self.OFF + r0
        return m[p // 8: (p + nw + 7) // 8 + 1].cpu().numpy(), p % 8

    def _cmp(self, j, c0, r0, nw, w, exp_out, exp_val):
        import numpy as np
        got = self.outs[j][r0 * w: (r0 + nw) * w].cpu().numpy()
        assert np.array_equal(got, exp_out[: nw * w]), f"parity: C5 vector payload of column {j} differs (chunk {c0}..)"
        nwords = (nw + 63) // 64
        got_v = self.vals[j][c0 * 256: c0 * 256 + nwords * 8].cpu().numpy().view(np.uint64)
        assert np.array_equal(got_v, exp_val[:nwords]), f"parity: C5 validity masks of column {j} differ (chunk {c0}..)"


def torch_uint8():
    import torch
    return torch.uint8


# ----------------------------------------------------------------------------- CPU baselines (oracle = the thing timed)
def cpu_reference_pass(batch, split=None):
    """The reference path on one result: duckdb_mb_arrow_get_column_* per column (the getter the
    schema's type_id selects, src/duckdb_native.c:2314-2339) + the MoonBit decoder loops.
    Returns seconds; split (a dict) receives the seconds spent in the C getters ("getters_s": what produces the Bytes)
    and in the decoders ("decode_s")."""
    import numpy as np
    import oracle
    from duckdb_mbt_b200 import chunks as ch
    t0 = time.perf_counter()
    ora = oracle.OracleResult(batch)
    tg = td = 0.0
    for j, col in enumerate(batch.columns):
        if col.type_id in (ch.T_TINYINT, ch.T_SMALLINT, ch.T_INTEGER):
            kind, dec = "int32", oracle.decode_int32
        elif col.type_id == ch.T_BIGINT:
            kind, dec = "int64", oracle.decode_int64_as_int
        elif col.type_id in (ch.T_FLOAT, ch.T_DOUBLE):
            kind, dec = "double", oracle.decode_double
        elif col.type_id == ch.T_BOOLEAN:
            kind, dec = "bool", oracle.decode_bool
        else:  # everything else is "string" in the reference's schema: duckdb_value_varchar per cell
            kind, dec = "string", None
        t1 = time.perf_counter()
        blob = ora.get_column(kind, j, True)
        t2 = time.perf_counter()
        if dec is not None:
            dec(blob, True)
        else:
            n = max(len(blob), 1)
            buf = np.frombuffer(blob, dtype=np.uint8) if blob else np.zeros(1, np.uint8)
            starts, ends, valid = np.zeros(n, np.int64), np.zeros(n, np.int64), np.zeros(n, np.uint8)
            oracle.lib().ora_decode_string(buf.ctypes.data, len(blob), 1, starts.ctypes.data, ends.ctypes.data, valid.ctypes.data)
        tg += t2 - t1
        td += time.perf_counter() - t2
    ora.close()
    if split is not None:
        split["getters_s"] = split.get("getters_s", 0.0) + tg
        split["decode_s"] = split.get("decode_s", 0.0) + td
    return time.perf_counter() - t0


def _cpu_worker(args):
    rows, seed, passes = args
    from duckdb_mbt_b200 import chunks as ch
    import oracle
    oracle.lib()
    batch = ch.config_c2(rows, seed=seed)
    split = {}
    times = [cpu_reference_pass(batch, split) for _ in range(passes)]
    return times, split


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation (oracle port) on the host cores."""
    if rank != 0:
        return
    import concurrent.futures as cf
    import oracle
    oracle.build()
    cores = max(1, min(os.cpu_count() or 1, env_int("DMB_REF_PROCS", 64)))
    rows = min(args.rows, CPU_SAMPLE_ROWS)
    passes = args.warmup + args.steps
    with cf.ProcessPoolExecutor(max_workers=cores) as ex:
        t0 = time.perf_counter()
        results = list(ex.map(_cpu_worker, [(rows, 20260103 + i, passes) for i in range(cores)]))
        wall = time.perf_counter() - t0
    # every worker converts its own <= 1M-row result `steps` times; aggregate over the timed passes
    per_worker = [sum(t[args.warmup:]) for t, _ in results]
    slowest = max(per_worker)
    value = cores * rows * args.steps / slowest
    getters_s = max(sp.get("getters_s", 0.0) for _, sp in results) * args.steps / passes
    decode_s = max(sp.get("decode_s", 0.0) for _, sp in results) * args.steps / passes
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * slowest / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "BASELINE.json configs[1]: lineitem-shaped table (4 INTEGER, 4 DECIMAL(15,2), 3 DATE, 5 VARCHAR) -> "
                               "reference packed getters + MoonBit decoders", "rows_per_step": cores * rows,
                   "note": "reference = CPU oracle port of src/duckdb_native.c:2357-2797 + src/duckdb_arrow_native.mbt:430-822 "
                           "(MoonBit + libduckdb cannot be built in this image); one <=1M-row result per process (the decoders' cap), "
                           f"{cores} processes (every host core the box gives)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{cores} processes x {rows} rows x {args.steps} steps of the C2 table, generation untimed"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": wall,
        # the same surface bench.py's e2e_getters leg times on the GPU arm, split the same way
        "getters_split": {"getters_only_rows_per_s": cores * rows * args.steps / max(getters_s, 1e-9),
                          "getters_ms_per_step": 1e3 * getters_s / args.steps, "decode_ms_per_step": 1e3 * decode_s / args.steps,
                          "note": "getters = the C stub's per-cell loops that produce the Bytes blobs (equal outputs to the GPU arm's "
                                  "c_abi_only figure, minus materialise); decode = the MoonBit decoder loops"},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- host-side input shapes for the e2e legs
def duckdb_layout_batch(hb, pad=4160):
    """The input the glue really hands over (INTEGRATION.md; src/duckdb_native.c:529-530,547,597-603): every 2048-row
    vector at its own address in PAGEABLE memory (never address-contiguous with its neighbours), validity masks likewise,
    and per-chunk string heaps that nobody registered (heap_len = 0, no inline-only hint)."""
    import numpy as np
    from duckdb_mbt_b200 import chunks as ch
    nch = hb.nchunks
    cols = []
    keep = []
    for col in hb.columns:
        w = col.width
        stride = VS * w + pad
        buf = np.empty(nch * stride, dtype=np.uint8)
        view = buf.reshape(nch, stride)[:, : VS * w]
        view[:] = col.data[: nch * VS * w].reshape(nch, VS * w)
        data_off = np.arange(nch, dtype=np.uint64) * np.uint64(stride)
        validity, val_off = None, np.full(nch, -1, dtype=np.int64)
        if col.validity is not None:
            vstride = (256 + pad) // 8
            validity = np.zeros(nch * vstride, dtype=np.uint64)
            validity.reshape(nch, vstride)[:, :32] = np.asarray(col.validity).reshape(-1)[: nch * 32].reshape(nch, 32)
            val_off = np.where(np.asarray(col.val_off) >= 0, np.arange(nch, dtype=np.int64) * vstride, -1)
        if col.phys == ch.P_STRING and col.heap is not None:
            ent = view.reshape(nch, VS, 16)
            lens = ent[:, :, 0:4].copy().view(np.uint32).reshape(nch, VS)
            ptrs = ent[:, :, 8:16].copy().view(np.uint64).reshape(nch, VS)
            isp = lens > 12
            old_base = np.uint64(col.heap.ctypes.data)
            gap = 64
            heap = np.empty(col.heap.shape[0] + nch * gap + 64, dtype=np.uint8)
            # the heap is in row order, so chunk k's strings are one span of it: move span k by k * gap bytes
            rel = np.where(isp, ptrs - old_base, np.uint64(0))
            lo = np.where(isp, rel, np.uint64(2**62)).min(axis=1)
            hi = np.where(isp, rel + lens.astype(np.uint64), np.uint64(0)).max(axis=1)
            for k in np.flatnonzero(hi > lo):
                a, b = int(lo[k]), int(hi[k])
                heap[a + k * gap: b + k * gap] = col.heap[a:b]
            shift = (np.arange(nch, dtype=np.uint64) * np.uint64(gap))[:, None]
            new = rel + shift + np.uint64(heap.ctypes.data)
            ent8 = ent[:, :, 8:16]
            ent8[isp] = new[isp].view(np.uint8).reshape(-1, 8)
            keep.append(heap)
        cols.append(ch.Column(col.name, col.type_id, col.phys, buf, data_off, validity, val_off, col.dec_width, col.dec_scale, None))
    out = ch.ChunkBatch(np.asarray(hb.counts, dtype=np.uint32).copy(), cols)
    out._keep = keep
    return out


# ----------------------------------------------------------------------------- ours
def run_ours(args, rank, local_rank, world):
    import numpy as np
    import torch
    import torch.distributed as dist

    from duckdb_mbt_b200 import arrow_result as ar
    from duckdb_mbt_b200 import chunks as ch
    from duckdb_mbt_b200 import devgen
    from duckdb_mbt_b200 import native as nat
    from duckdb_mbt_b200 import pinned
    from duckdb_mbt_b200 import shard
    from duckdb_mbt_b200.appender import _release as ap_release

    nat.lib()  # fails loudly when libduckdb_mb_gpu.so is missing: no fallback
    bind_to_gpu_numa_node(local_rank)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    def reduce_ranks(xs, op):
        if world == 1:
            return list(xs)
        t = torch.tensor(list(xs), dtype=torch.float64, device=device)
        dist.all_reduce(t, op=op)
        return [float(v) for v in t.tolist()]

    def max_over_ranks(x: float) -> float:
        return reduce_ranks([x], dist.ReduceOp.MAX)[0]

    n = args.rows
    e2e_rows = min(n, args.e2e_rows)
    steps, warmup = args.steps, args.warmup
    side_steps = max(1, min(steps, 5))  # the other configs / legs: fewer steps keep the default run within minutes
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_gbs, peak_src = (float(peaks["hbm_gbs"]), "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (6650.0, "fallback")
    do_parity = not args.no_parity
    if do_parity:
        import oracle
        oracle.build()

    # ---- inputs: generated in HBM; the e2e leg gets the same bytes in page-locked host slabs
    pinned_arrays = []

    def host_heap_alloc(nbytes):
        a = pinned.pinned_empty(nbytes)
        pinned_arrays.append(a)
        return a

    t_setup = time.perf_counter()
    db = build_c2_device(n, 20260103 + rank, device, host_heap_alloc=host_heap_alloc if e2e_rows == n else None)
    step = DeviceStep(db)
    torch.cuda.synchronize(device)

    # ---- parity first (BASELINE.md §2.3): sampled windows of every output column against the oracle, then warm-up
    parity = {}
    step.run()
    step.check()
    if do_parity:
        parity["C2"] = parity_check_step(step, seed=1 + rank)
    for _ in range(warmup):
        step.run()
    step.check()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    # ---- value: device-resident, CUDA events on the launching (current) stream
    spans = []
    barrier()
    ev_a, ev_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev_a.record()
    for _ in range(steps):
        spans.append(step.run(record=True))
    ev_b.record()
    barrier()
    dev_ms = ev_a.elapsed_time(ev_b)
    step.check()
    if args.dump_outputs and rank == 0:
        files = dump_step_outputs(step, args.dump_outputs)
        print(f"bench.py: {len(files)} arrays of the last timed step written to {args.dump_outputs}", file=sys.stderr, flush=True)
    fixed_ms = sum(sp[0].elapsed_time(sp[1]) for sp in spans) / steps
    string_ms = sum(sp[1].elapsed_time(sp[2]) for sp in spans) / steps
    string_cols = [db.batch.columns[so.col].name for so in step.strings]
    string_col_ms = {}
    for ci, nm in enumerate(string_cols):
        string_col_ms[nm] = sum((sp[1] if ci == 0 else sp[3][ci - 1]).elapsed_time(sp[3][ci]) for sp in spans) / steps
    nd = db.nrows
    string_col_alg = {db.batch.columns[so.col].name: 16 * nd + db.meta[so.col]["ptr_len"] + 4 * (nd + 1) + db.meta[so.col]["total_len"]
                      for so in step.strings}
    # which kernel a VARCHAR column goes to (kernels_string.cu, dmb_dev_string_batch): the persistent TMA pipeline
    # string_pack_kernel; columns without a heap take its lean form (template argument HEAP = false), reported as a family
    # of its own -- or the one-CTA-per-tile string_short_kernel when DMB_STR_SHORT_RPT selects it (A/B knob)
    noheap_kernel = "string_short_kernel" if int(os.environ.get("DMB_STR_SHORT_RPT", "0") or 0) > 0 else "string_pack_kernel<no heap>"
    string_col_kernel = {db.batch.columns[so.col].name: (noheap_kernel if db.meta[so.col]["ptr_len"] == 0 else "string_pack_kernel")
                         for so in step.strings}
    string_totals = [float(db.meta[so.col]["total_len"]) for so in step.strings]
    dev_ms_max = max_over_ranks(dev_ms)
    value = world * n * steps / (dev_ms_max / 1e3)
    step_alg_fixed, step_alg_string = step.alg_fixed, step.alg_string
    alg_bytes = step_alg_fixed + step_alg_string
    n_fixed_launches = step.n_fixed_launches
    n_launches = step.launches
    # one table over N GPUs (SURVEY.md §8e): the only cross-GPU datum is one byte total per string column per GPU;
    # an exclusive scan of those on the host gives the base every GPU's offsets are shifted by
    sharded_table = None
    if world > 1:
        t = torch.tensor(string_totals, dtype=torch.float64, device=device)
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        per_gpu = [[int(v) for v in x.tolist()] for x in allt]
        sharded_table = {"rows": world * n, "string_columns": string_cols,
                         "offset_bases_per_gpu": [shard.string_bases([per_gpu[g][ci] for g in range(world)]) for ci in range(len(string_cols))]}

    # ---- the other BASELINE configs, device-resident, same clock-sampled region (C2 stays resident for the e2e legs)
    configs = {}

    def time_steps(run, k, flush=None):
        """k timed steps; with `flush` (a device buffer larger than L2) written between them when the working set is small"""
        evs = []
        for _ in range(k):
            if flush is not None:
                flush.add_(1)
            evs.append(run(record=True))
        torch.cuda.synchronize(device)
        return evs

    def add_config(name, rows_per_gpu, rows_total_all, evs, k, alg, split, extra):
        ms = sum(e[0].elapsed_time(e[2]) for e in evs) / k
        ms_max = max_over_ranks(ms)
        configs[name] = {"rows": rows_total_all, "rows_per_gpu": rows_per_gpu, "ms": ms_max, "rows_per_s": rows_total_all / ms_max * 1e3,
                         "gb_per_s": alg / 1e6 / ms, "frac": alg / 1e6 / ms / peak_gbs, "algorithmic_bytes_per_gpu": alg,
                         "kernel_split": split, "steps": k, **extra}
        if do_parity:
            configs[name]["parity_checked_rows"] = parity.get(name)

    def split_of(evs, k, alg_a, alg_b, name_a, name_b):
        a = sum(e[0].elapsed_time(e[1]) for e in evs) / k
        b = sum(e[1].elapsed_time(e[2]) for e in evs) / k
        out = {}
        if alg_a:
            out[name_a] = {"ms": a, "gb_per_s": alg_a / 1e6 / a, "frac": alg_a / 1e6 / a / peak_gbs}
        if alg_b:
            out[name_b] = {"ms": b, "gb_per_s": alg_b / 1e6 / b, "frac": alg_b / 1e6 / b / peak_gbs}
        return out

    if not args.no_configs:
        # C1: the reference's own CPU-runnable case, 1 M rows x 3 columns = 32.75 MB per pass (launch bound; L2 flushed)
        c1 = devgen.GeneratedBatch(1_000_000, device)
        g = torch.Generator(device=device)
        g.manual_seed(20260102 + rank)
        c1.add_fixed(ch.T_INTEGER, 0, g, 0.0, "CAST(i AS INTEGER)", lo=0, hi=1_000_000)
        c1.add_fixed(ch.T_DOUBLE, 0, g, 0.0, "CAST(i AS DOUBLE)")
        c1.add_fixed(ch.T_INTEGER, 0, g, 1.0, "CASE")  # every row NULL
        s1 = DeviceStep(c1)
        s1.run()
        if do_parity:
            parity["C1"] = parity_check_step(s1, seed=2)
        flush = torch.zeros(256 << 20, dtype=torch.uint8, device=device)
        for _ in range(3):
            s1.run()
        evs = time_steps(s1.run, side_steps, flush=flush)
        add_config("C1", 1_000_000, world * 1_000_000, evs, side_steps, s1.alg_fixed, split_of(evs, side_steps, s1.alg_fixed, 0, "fixed_batch_kernel", ""),
                   {"workload": "BASELINE.json configs[0]: range(1000000) -> INTEGER, DOUBLE, all-NULL CASE; 32.75 MB per pass: launch-latency bound, "
                                "not an HBM number", "l2": "256 MB written between timed steps (working set < L2)", "launches": s1.launches})
        del c1, s1, flush, evs

        # C3: 100 M VARCHAR rows, len U[0,64], 10 % NULL: > 2^31 string bytes -> int64 offsets
        n3 = args.c3_rows
        c3 = devgen.string_batch(n3, seed=20260104 + rank, null_frac=0.10, max_len=64, device=device)
        large = c3.total_len > 2**31 - 1
        s3 = DeviceStep(c3, large=large)
        s3.run()
        s3.check()
        if do_parity:
            parity["C3"] = parity_check_step(s3, seed=3)
        for _ in range(3):
            s3.run()
        evs = time_steps(s3.run, side_steps)
        s3.check()
        alg3 = s3.alg_fixed + s3.alg_string
        add_config("C3", n3, world * n3, evs, side_steps, alg3,
                   split_of(evs, side_steps, s3.alg_fixed, s3.alg_string, "fixed_batch_kernel(validity)", "string_pack_kernel"),
                   {"workload": "BASELINE.json configs[2]: VARCHAR len U[0,64], 20% inline / 80% pointer, 10% NULL -> Arrow "
                                + ("large_utf8 (int64 offsets: > 2^31 string bytes)" if large else "utf8"),
                    "utf8_bytes": c3.total_len, "launches": s3.launches})
        del c3, s3, evs
        torch.cuda.empty_cache()

        # C4: 64 columns (22 TIMESTAMP, 21 DECIMAL(18,3) -> decimal128, 21 HUGEINT), 30 % NULL; row groups sharded over the GPUs
        n4 = args.c4_rows // world
        cols4 = [(ch.T_TIMESTAMP, 0)] * 22 + [(ch.T_DECIMAL, 18)] * 21 + [(ch.T_HUGEINT, 0)] * 21
        c4 = devgen.fixed_batch(n4, cols4, null_frac=0.30, seed=20260105 + rank, device=device)
        for c in c4.batch.columns:
            if c.type_id == ch.T_DECIMAL:
                c.dec_scale = 3
        s4 = DeviceStep(c4)
        s4.run()
        if do_parity:
            parity["C4"] = parity_check_step(s4, seed=4, k=0)
        for _ in range(3):
            s4.run()
        evs = time_steps(s4.run, side_steps)
        add_config("C4", n4, world * n4, evs, side_steps, s4.alg_fixed, split_of(evs, side_steps, s4.alg_fixed, 0, "fixed_batch_kernel", ""),
                   {"workload": "BASELINE.json configs[3]: 64 columns (22 TIMESTAMP, 21 DECIMAL(18,3)->decimal128, 21 HUGEINT), 30% NULL, garbage "
                                f"under NULLs; {args.c4_rows} rows sharded over {world} GPU(s) (strong scaling)", "launches": s4.launches})
        del c4, s4, evs
        torch.cuda.empty_cache()

        # C5: reverse path, 500 M rows over the GPUs, converted in device-resident batches of <= 50 M rows, timed as a whole
        rows5 = args.c5_rows // world
        nb5 = max(1, -(-rows5 // 50_000_000))
        batch5 = rows5 // nb5
        s5 = ReverseStep(batch5, 20260106 + rank, device)
        s5.run()
        if do_parity:
            parity["C5"] = s5.parity_check(seed=5)
        for _ in range(2):
            s5.run()

        def run5(record=False):
            first = None
            for _ in range(nb5):
                e = s5.run(record=record)
                first = first or e
            return (first[0], first[1], e[2]) if record else None

        k5 = max(1, min(side_steps, 3))
        evs = time_steps(run5, k5)
        ms5 = sum(e[0].elapsed_time(e[2]) for e in evs) / k5
        one = s5.run(record=True)
        torch.cuda.synchronize(device)
        alg5 = nb5 * (s5.alg_fixed + s5.alg_string)
        ms5_max = max_over_ranks(ms5)
        configs["C5"] = {"rows": world * nb5 * batch5, "rows_per_gpu": nb5 * batch5, "ms": ms5_max, "rows_per_s": world * nb5 * batch5 / ms5_max * 1e3,
                         "gb_per_s": alg5 / 1e6 / ms5, "frac": alg5 / 1e6 / ms5 / peak_gbs, "algorithmic_bytes_per_gpu": alg5, "steps": k5,
                         "kernel_split": split_of([one], 1, s5.alg_fixed, s5.alg_string, "rev_fixed_kernel", "rev_string_kernel"),
                         "workload": f"BASELINE.json configs[4]: Arrow (int32,int64,float64,bool,utf8 U[0,24]) -> DataChunk vectors, 10% NULL, bit offset 3; "
                                     f"{args.c5_rows} rows over {world} GPU(s) = {nb5} batch(es) of {batch5} rows per GPU, timed as a whole",
                         "batches_per_gpu": nb5, "launches": nb5 * 5}
        if do_parity:
            configs["C5"]["parity_checked_rows"] = parity.get("C5")
        del s5, evs, one
        torch.cuda.empty_cache()

    # ---- beyond BASELINE.json's configs (SURVEY.md 8f item 3), inside the same clock-sampled region: LIST<INTEGER> -> Arrow
    # list<int32> and ENUM -> utf8 at the device API (profiles/bench_configs.py builds the inputs in HBM; the ENUM output is
    # compared bit for bit with the two-step path, the LIST totals with the generator's)
    if not args.no_configs:
        sys.path.insert(0, os.path.join(ROOT, "profiles"))
        import bench_configs as bc
        bc.QUIET = True
        for name, fn, kernel in (("LIST", bc.clist, "list_emit_kernel"), ("ENUM", bc.cenum, "enum_pack_kernel")):
            torch.cuda.empty_cache()
            fn(1.0, None)
            ln = bc.LINES[-1]
            ms_max = max_over_ranks(ln["ms"])
            configs[name] = {"rows": world * ln["rows"], "rows_per_gpu": ln["rows"], "ms": ms_max, "rows_per_s": world * ln["rows"] / ms_max * 1e3,
                             "gb_per_s": ln["gb_per_s"], "frac": ln["gb_per_s"] / peak_gbs, "algorithmic_bytes_per_gpu": int(ln["alg_GB"] * 1e9),
                             "kernel_split": {kernel: {"ms": ln["ms"], "gb_per_s": ln["gb_per_s"], "frac": ln["gb_per_s"] / peak_gbs}},
                             "steps": 5, "workload": "beyond BASELINE.json (SURVEY.md 8f item 3), per GPU: " + ln["config"], "launches": 1,
                             **{k_: v_ for k_, v_ in ln.items() if k_ in ("child_elements", "two_step_ms", "enum_to_string_t_kernel_ms", "heap_less_string_kernel_ms")}}
        torch.cuda.empty_cache()

    # ---- e2e: host API, page-locked host buffers, H2D + kernels + D2H timed
    if e2e_rows != n:
        del step, db
        torch.cuda.empty_cache()
        db = build_c2_device(e2e_rows, 20260103 + rank, device, host_heap_alloc=host_heap_alloc)

    def alloc(nb):
        a = pinned.pinned_empty(nb)
        pinned_arrays.append(a)
        return a

    host_batch = db.to_host_batch(alloc=alloc)
    del db
    if e2e_rows == n:
        del step
    torch.cuda.empty_cache()
    setup_s = time.perf_counter() - t_setup
    link = measure_host_link(device, barrier)
    ctx = ar.GpuContext(local_rank)

    def e2e_leg(hb, k, w):
        """k timed calls of from_chunks + materialise + export of the whole record batch"""
        def one():
            h = ctx.lib.duckdb_mb_gpu_result_from_chunks(ctx.handle, C.byref(hb.struct))
            if not h:
                raise RuntimeError(nat.last_error())
            res = ar.ArrowResult(ctx, h, hb)
            res.materialise()
            arr, sch = res.export_c(-1)  # the step's result: one record batch in page-locked host memory
            rows_out = arr.length
            t = res.timings()
            ap_release(arr)
            ap_release(sch)
            res.close()
            return rows_out, t
        for _ in range(max(w, 1)):
            rows_out, t = one()
            assert rows_out == e2e_rows
        barrier()
        t0 = time.perf_counter()
        kernels_ms = 0.0
        for _ in range(k):
            rows_out, t = one()
            kernels_ms += t["kernels_ms"]
        ctx.sync()
        secs = time.perf_counter() - t0
        barrier()
        secs_max = max_over_ranks(secs)
        link_gbs = (t["h2d_bytes"] + t["d2h_bytes"]) * k / secs / 1e9
        return {"value": world * e2e_rows * k / secs_max, "unit": UNIT, "h2d_bytes_per_step": int(t["h2d_bytes"]),
                "d2h_bytes_per_step": int(t["d2h_bytes"]), "ms_per_step": 1e3 * secs_max / k, "steps": k,
                "link_gb_per_s_per_gpu": link_gbs, "link_frac": link_gbs / link["bidir_sum_gbs"] if link.get("bidir_sum_gbs") else None,
                "kernels_ms_per_step": kernels_ms / k}

    hb = ar.HostBatch(host_batch, pinned=True)
    e2e = e2e_leg(hb, steps, warmup)
    e2e["host_link_measured"] = link
    e2e["host_buffers"] = "page-locked (DMB_BATCH_PINNED), contiguous chunk slabs, registered contiguous heaps"
    e2e["aggregate_link_gb_per_s"] = e2e["link_gb_per_s_per_gpu"] * world
    del hb

    # ---- e2e on the layout the integration delivers, and the reference's own getter surface
    e2e_layout = None
    e2e_getters = None
    need_gb = 2.2 * e2e_rows * 180 / 1e9
    if not args.no_layout_leg and mem_available_gb() > need_gb + 8:
        t_l = time.perf_counter()
        layout = duckdb_layout_batch(host_batch)
        hb2 = ar.HostBatch(layout, pinned=False, register_heap=False)
        e2e_layout = e2e_leg(hb2, side_steps, 2)
        e2e_layout["host_buffers"] = ("pageable; one buffer per 2048-row vector at its own address; per-chunk string heaps, not registered "
                                      "(heap_len = 0: the stager compacts the pointed-to bytes); flags = 0; no inline-only hint")
        e2e_layout["vs_pinned_leg"] = e2e_layout["value"] / e2e["value"]
        e2e_layout["build_s"] = time.perf_counter() - t_l
        # the reference's surface on <= 1 M-row results (its decoders' cap): from_chunks + 16 nullable getters + decoder mirror
        n_res = 16
        per = GETTER_CHUNKS
        getter_of = {ch.T_INTEGER: "int32", ch.T_TINYINT: "int32", ch.T_SMALLINT: "int32", ch.T_BIGINT: "int64", ch.T_FLOAT: "double",
                     ch.T_DOUBLE: "double", ch.T_BOOLEAN: "bool"}
        subs = [ar.HostBatch(shard.slice_batch(layout, i * per, (i + 1) * per), pinned=False, register_heap=False)
                for i in range(min(n_res, layout.nchunks // per))]
        rows_res = sum(s.batch.nrows for s in subs)

        import concurrent.futures as cf
        tsplit = {"from_chunks_s": 0.0, "c_getters_s": 0.0, "decode_s": 0.0}
        pool = cf.ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 1))
        fixed_fmt = {"int32": (4, "<i4"), "int64": (8, "<i8"), "double": (8, "<f8"), "bool": (1, np.uint8)}

        def decode_one(res, kind, blob):
            with blob as view:  # the decoder mirror (MoonBit-side work in the reference): numpy releases the GIL, columns decode in parallel
                if kind == "string":
                    return int(ar.decode_string_spans(view, True)[2].shape[0])
                w, dt = fixed_fmt[kind]
                return int(res._decode_fixed(view, w, np.dtype(dt), True)[1].shape[0])

        def getters_step():
            """results one after the other through the C ABI; the decoder mirror of result i runs on the pool while the C ABI
            converts result i + 1 (decode_s = the time the caller still had to wait for decoders)"""
            got = 0
            pending = None

            def finish(p):
                res_p, futs = p
                t = time.perf_counter()
                n_ = sum(f.result() for f in futs)
                tsplit["decode_s"] += time.perf_counter() - t
                res_p.close()
                return n_

            for s in subs:
                t0 = time.perf_counter()
                h = ctx.lib.duckdb_mb_gpu_result_from_chunks(ctx.handle, C.byref(s.struct))
                res = ar.ArrowResult(ctx, h, s)
                t1 = time.perf_counter()
                tsplit["from_chunks_s"] += t1 - t0
                blobs = []
                for j, col in enumerate(s.batch.columns):  # the C-ABI calls, one at a time like the reference's FFI
                    kind = getter_of.get(col.type_id, "string")
                    blobs.append((kind, res._blob(kind, j, True)))
                tsplit["c_getters_s"] += time.perf_counter() - t1
                futs = [pool.submit(decode_one, res, kb[0], kb[1]) for kb in blobs]
                if pending is not None:
                    got += finish(pending)
                pending = (res, futs)
            if pending is not None:
                got += finish(pending)
            return got

        assert getters_step() == rows_res * len(layout.columns)
        getters_step()
        barrier()
        t0 = time.perf_counter()
        kg = max(1, min(side_steps, 3))
        for k_ in tsplit:
            tsplit[k_] = 0.0
        for _ in range(kg):
            getters_step()
        secs = max_over_ranks(time.perf_counter() - t0)
        barrier()
        e2e_getters = {"value": world * rows_res * kg / secs, "unit": UNIT, "ms_per_step": 1e3 * secs / kg, "steps": kg,
                       "rows_per_step_per_gpu": rows_res, "results_per_step": len(subs),
                       "ms_per_step_split": {k_: 1e3 * v_ / kg for k_, v_ in tsplit.items()},
                       "c_abi_only_rows_per_s": world * rows_res * kg / max(tsplit["from_chunks_s"] + tsplit["c_getters_s"], 1e-9),
                       "what": "per <= 1 M-row result (the reference decoders' cap): duckdb_mb_gpu_result_from_chunks on the DuckDB "
                               "layout + the 16 duckdb_mb_arrow_get_column_*_nullable getters the schema selects + the decoder mirror "
                               "(arrow_result.py, columns decoded on a thread pool while the C ABI converts the next result) -- the surface "
                               "--impl reference times on the CPU"}
        pool.shutdown()
        del subs, hb2, layout
    elif not args.no_layout_leg:
        e2e_layout = {"skipped": f"host has {mem_available_gb():.0f} GB available, the leg needs ~{need_gb:.0f} GB more"}
    clocks = sampler.stop() if rank == 0 else None  # sampled from the start of the device-timed region to the end of the e2e legs

    # ---- cpu baselines (rank 0, N=1 only): reference-equivalent port on 1 core; columnar OpenMP on all cores
    cpu = None
    cpu_col = None
    if rank == 0 and world == 1 and not args.no_cpu:
        import oracle
        oracle.build()
        sample = min(n, CPU_SAMPLE_ROWS)
        cb = shard.slice_batch(host_batch, 0, -(-sample // VS))
        secs = cpu_reference_pass(cb)
        cpu = {"value": cb.nrows / secs, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": f"{cb.nrows} rows of the C2 table, one result (the reference decoders' 1M-row cap), "
                         f"{secs:.2f} s: materialise + 16 packed getters + MoonBit decoder loops"}
        try:
            from oracle import columnar
            crow = min(e2e_rows, 8_000_000)
            cbatch = shard.slice_batch(host_batch, 0, -(-crow // VS))
            conv = columnar.ColumnarConverter(cbatch, threads=os.cpu_count())
            conv.run()
            ts = [conv.run() for _ in range(3)]
            best = min(ts)
            cpu_col = {"value": cbatch.nrows / best, "unit": UNIT, "cores": conv.threads, "kind": "columnar-openmp",
                       "sample": f"{cbatch.nrows} rows of the C2 table -> Arrow buffers (16 columns), best of 3 passes of {best * 1e3:.0f} ms, "
                                 "outputs preallocated; gcc -O3 -march=native -fopenmp (oracle/columnar.c), checked against the oracle in tests/"}
            del conv
        except Exception as e:  # the strong-CPU line is context, never a reason to lose the run
            cpu_col = {"unavailable": str(e)[:200]}
    ctx.close()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- roofline of the dominant kernel: the family with the most device time in a step
    families = {"fixed_batch_kernel": [fixed_ms, step_alg_fixed, n_fixed_launches]}
    for nm, k in string_col_kernel.items():
        f = families.setdefault(k, [0.0, 0, 0])
        f[0] += string_col_ms[nm]
        f[1] += string_col_alg[nm]
        f[2] += 1
    dominant = max(families, key=lambda k: families[k][0])
    dom_ms, dom_alg, dom_launches = families[dominant]
    achieved = dom_alg / 1e6 / dom_ms  # GB/s: algorithmic bytes of the kernel's launches in a step / their device time
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if tj.get("rows") == n and dominant in tj.get("kernels", {}):
            traffic = tj["kernels"][dominant].get("dram_bytes_per_launch")
    except Exception:
        pass
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": dev_ms_max / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": "BASELINE.json configs[1]: synthetic lineitem-shaped table (4 INTEGER, 4 DECIMAL(15,2)->decimal128, "
                               "3 DATE, 5 VARCHAR: returnflag, linestatus, shipinstruct, shipmode, comment U[10,43]; no NULLs) "
                               "-> Arrow record batch",
                   "rows_per_gpu": n, "chunks_per_gpu": (n + 2047) // 2048, "parallelism": f"row-group shards x{world}, no collective",
                   "l2": "inputs (~10.5 GB per GPU at 60M rows) far exceed the 126 MB L2: no flush between steps",
                   "string_heap": "one contiguous heap per VARCHAR column, registered with the batch; pointers rebased in-kernel",
                   "e2e_rows_per_gpu": e2e_rows, "sharded_table": sharded_table},
        "gb_per_s": world * alg_bytes * steps / (dev_ms_max / 1e3) / 1e9,
        "algorithmic_bytes_per_step_per_gpu": alg_bytes,
        "hbm_frac_whole_step": alg_bytes * steps / (dev_ms / 1e3) / 1e9 / peak_gbs,
        "parity_checked_rows": (sum(v for v in parity.values() if v) if do_parity else 0),
        "parity": ({"checked_before_timing": True, "cells_per_config": parity,
                    "how": "sampled windows of ~1 M rows (head, ragged tail, seeded random) of every output column, bit-exact vs the CPU oracle"}
                   if do_parity else {"checked_before_timing": False}),
        "e2e": e2e,
        "e2e_duckdb_layout": e2e_layout,
        "e2e_getters": e2e_getters,
        "configs": configs,
        "roofline": {"bound": "hbm", "kernel": dominant, "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
                     "frac": achieved / peak_gbs, "traffic": traffic, "peak_source": peak_src,
                     "launches_per_step": dom_launches, "algorithmic_bytes_per_launch": dom_alg / dom_launches,
                     "avg_launch_ms": dom_ms / dom_launches},
        "cpu_baseline": cpu,
        "cpu_columnar": cpu_col,
        "gpu_launches": n_launches * steps,
        "clocks": clocks,
        "kernel_ms_per_step": {**{k: v[0] for k, v in families.items()},
                               "families": {k: {"ms": v[0], "launches": v[2], "gb_per_s": v[1] / 1e6 / v[0], "frac": v[1] / 1e6 / v[0] / peak_gbs}
                                            for k, v in families.items()},
                               "string_ms": string_ms, "string_gb_per_s": step_alg_string / 1e6 / string_ms,
                               "string_columns": {nm: {"kernel": string_col_kernel[nm], "ms": string_col_ms[nm],
                                                       "gb_per_s": string_col_alg[nm] / 1e6 / string_col_ms[nm]}
                                                  for nm in string_col_ms}},
        "setup_s": setup_s,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=env_int("DMB_BENCH_ROWS", DEFAULT_ROWS), help="rows per GPU")
    ap.add_argument("--e2e-rows", type=int, default=env_int("DMB_BENCH_E2E_ROWS", DEFAULT_ROWS), help="rows per GPU for the host-buffer leg")
    ap.add_argument("--c3-rows", type=int, default=env_int("DMB_BENCH_C3_ROWS", 100_000_000), help="C3 rows per GPU")
    ap.add_argument("--c4-rows", type=int, default=env_int("DMB_BENCH_C4_ROWS", 10_000_000), help="C4 rows, sharded over the GPUs")
    ap.add_argument("--c5-rows", type=int, default=env_int("DMB_BENCH_C5_ROWS", 500_000_000), help="C5 rows, sharded over the GPUs")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / cpu_columnar legs")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle comparison before timing")
    ap.add_argument("--no-configs", action="store_true", help="skip C1 / C3 / C4 / C5")
    ap.add_argument("--no-layout-leg", action="store_true", help="skip e2e_duckdb_layout / e2e_getters")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a seeded row sample of what the last one "
                                                          "computed (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl ours")
    rank = env_int("RANK", 0)
    local_rank = env_int("LOCAL_RANK", 0)
    world = env_int("WORLD_SIZE", 1)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
