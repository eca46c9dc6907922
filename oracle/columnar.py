"""ctypes loader + driver for oracle/columnar.c: the all-core columnar CPU line (SURVEY.md §8d, BASELINE.md §2.2).
TEST / BENCH INFRASTRUCTURE ONLY (tests/ and bench.py's cpu_baseline leg)."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile
import time
from typing import List, Optional

import numpy as np

from . import OraBatch, OraColumn, _ptr

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def _cpu_tag() -> str:
    """-march=native code must not travel to a different CPU: one build per CPU model + flag set"""
    try:
        txt = open("/proc/cpuinfo").read()
        model = next((ln for ln in txt.splitlines() if ln.startswith("model name")), "")
        flags = next((ln for ln in txt.splitlines() if ln.startswith("flags")), "")
        return hashlib.sha1((model + flags).encode()).hexdigest()[:10]
    except OSError:
        return "generic"


def lib_path() -> str:
    return os.path.join(_HERE, f"libcolumnar.{_cpu_tag()}.so")


def _stale(out: str) -> bool:
    return not os.path.exists(out) or os.path.getmtime(out) < os.path.getmtime(os.path.join(_HERE, "columnar.c"))


def build(force: bool = False, out: Optional[str] = None) -> str:
    src, out = os.path.join(_HERE, "columnar.c"), out or lib_path()
    if force or _stale(out):
        err = None
        for cc in ("/usr/bin/gcc", "gcc", os.environ.get("CC", "cc")):  # (a wrapper gcc without libgomp.spec exists in this image)
            try:
                subprocess.check_call([cc, "-O3", "-march=native", "-fopenmp", "-fPIC", "-shared", "-std=gnu11", "-Wall", "-Wextra",
                                       "-o", out, src], stderr=subprocess.DEVNULL)
                err = None
                break
            except (OSError, subprocess.CalledProcessError) as e:
                err = e
        if err is not None:
            raise RuntimeError(f"cannot build oracle/columnar.c with OpenMP: {err}")
    return out


def lib():
    global _lib
    if _lib is None:
        if _stale(lib_path()):
            # not built in the tree for this CPU (the tree may be read-only): compile into a temporary directory, load, remove
            with tempfile.TemporaryDirectory(prefix="dmb_columnar_") as tmp:
                L = C.CDLL(build(out=os.path.join(tmp, os.path.basename(lib_path()))))
        else:
            L = C.CDLL(lib_path())
        L.col_fixed.restype = C.c_int64
        L.col_fixed.argtypes = [C.POINTER(OraBatch), C.c_int32, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.col_string.restype = C.c_int64
        L.col_string.argtypes = [C.POINTER(OraBatch), C.c_int32, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.POINTER(C.c_int64), C.c_int]
        L.col_max_threads.restype = C.c_int
        _lib = L
    return _lib


P_STRING, T_DECIMAL, T_HUGEINT = 14, 19, 16
PHYS_W = [1, 1, 2, 4, 8, 1, 2, 4, 8, 4, 8, 16, 16, 16, 16]


class ColumnarConverter:
    """DataChunk batch -> Arrow buffers on the host cores (outputs preallocated and pre-faulted: only the conversion is timed)."""

    def __init__(self, batch, threads: Optional[int] = None):
        L = lib()
        self.batch = batch
        self.threads = int(threads or os.cpu_count() or 1)
        self.counts = np.ascontiguousarray(batch.counts, dtype=np.uint32)
        self.row_off = np.zeros(self.counts.shape[0] + 1, dtype=np.int64)
        np.cumsum(self.counts, dtype=np.int64, out=self.row_off[1:])
        n = int(self.row_off[-1])
        self.nrows = n
        ncols = len(batch.columns)
        self._cols = (OraColumn * max(ncols, 1))()
        self._names = []
        self.out: List[dict] = []
        for i, c in enumerate(batch.columns):
            nm = c.name.encode()
            self._names.append(nm)
            self._cols[i] = OraColumn(c.type_id, c.phys, c.dec_width, c.dec_scale, _ptr(c.data), _ptr(c.data_off), _ptr(c.validity),
                                      _ptr(c.val_off), nm, None, None, 0)
            o = {"bitmap": np.zeros((n + 63) // 64 * 8, dtype=np.uint8)}
            if c.phys == P_STRING:
                heap = 0 if getattr(c, "heap", None) is None else int(c.heap.shape[0])
                o["large"] = 12 * n + heap > 0x7FFFFFFF
                o["offsets"] = np.zeros(n + 1, dtype=np.int64 if o["large"] else np.int32)
                o["data"] = np.zeros(12 * n + heap + 16, dtype=np.uint8)
                o["chunk_base"] = np.zeros(self.counts.shape[0] + 1, dtype=np.int64)
            else:
                widen = c.type_id == T_DECIMAL and c.phys != 11
                o["dst"] = 6 if widen else 0
                o["width"] = 16 if widen else PHYS_W[c.phys]
                o["values"] = np.zeros(n * o["width"], dtype=np.uint8)
            self.out.append(o)
        self._b = OraBatch(self.counts.shape[0], _ptr(self.counts), ncols, self._cols)
        self.L = L

    def run(self) -> float:
        """one conversion of every column; returns seconds"""
        L, b = self.L, C.byref(self._b)
        t0 = time.perf_counter()
        for i, (c, o) in enumerate(zip(self.batch.columns, self.out)):
            o["bitmap"][:] = 0
            if c.phys == P_STRING:
                nulls = C.c_int64(0)
                o["total"] = L.col_string(b, i, 1 if o["large"] else 0, _ptr(self.row_off), _ptr(o["offsets"]), _ptr(o["data"]),
                                          _ptr(o["bitmap"]), _ptr(o["chunk_base"]), C.byref(nulls), self.threads)
                o["nulls"] = nulls.value
            else:
                o["nulls"] = L.col_fixed(b, i, o["dst"], _ptr(self.row_off), _ptr(o["values"]), _ptr(o["bitmap"]), self.threads)
        return time.perf_counter() - t0
