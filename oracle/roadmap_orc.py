"""ctypes binding of the map-change / roadmap-update restatement (TEST INFRASTRUCTURE ONLY).

    oracle/roadmap_oracle.c -> liborc_roadmap.so   (processors::computeChange, the per-vertex / per-edge questions of
                                                    LazyPRMStarMinUpdateMaintainer, grid_map's LineIterator)

The library is compiled on first use with the flags of oracle/Makefile's port library (gcc -O2 -ffp-contract=off), into
oracle/ when that directory is writable and into the temporary directory otherwise.
Only tests/ and profiles/ may import this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "roadmap_oracle.c")
CFLAGS = ["-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra", "-Wno-unused-parameter"]

_lib = None


class OrcGrid(C.Structure):
    _fields_ = [("elevation", C.c_void_p), ("traversability_thresholded", C.c_void_p), ("rows", C.c_int),
                ("cols", C.c_int), ("res", C.c_double), ("cx", C.c_double), ("cy", C.c_double)]


def _so_path() -> str:
    d = HERE if os.access(HERE, os.W_OK) else tempfile.gettempdir()
    return os.path.join(d, "liborc_roadmap.so")


def build() -> str:
    """Compile liborc_roadmap.so if it is missing or older than its source; returns its path."""
    so = _so_path()
    if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(SRC):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.run([os.environ.get("CC", "gcc")] + CFLAGS + ["-shared", "-o", tmp, SRC, "-lm"], check=True)
        os.replace(tmp, so)
    return so


def _load():
    global _lib
    if _lib is None:
        lib = C.CDLL(build())
        lib.orc_compute_change.argtypes = [C.POINTER(OrcGrid), C.POINTER(OrcGrid), C.c_float, C.c_void_p, C.c_void_p]
        lib.orc_roadmap_updates.argtypes = [C.POINTER(OrcGrid), C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p,
                                            C.c_size_t, C.c_int, C.c_void_p, C.c_void_p]
        lib.orc_line_cells.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]
        _lib = lib
    return _lib


def _grid(m, keep):
    """OrcGrid of a map with `elevation` and `traversability_thresholded`."""
    ptrs = []
    for name in ("elevation", "traversability_thresholded"):
        a = np.asfortranarray(getattr(m, name), dtype=np.float32)
        keep.append(a)
        ptrs.append(a.ctypes.data)
    rows, cols = m.elevation.shape
    return OrcGrid(ptrs[0], ptrs[1], rows, cols, float(m.res), float(m.cx), float(m.cy))


def compute_change(map_new, map_old, thr: float):
    """processors::computeChange restated: (updated [rows_new, cols_new] float32 F-order, overlap_ok)."""
    lib = _load()
    keep = []
    gn, go = _grid(map_new, keep), _grid(map_old, keep)
    upd = np.empty((gn.rows, gn.cols), np.float32, order="F")
    ok = C.c_int(0)
    assert lib.orc_compute_change(C.byref(gn), C.byref(go), float(thr), upd.ctypes.data, C.byref(ok)) == 0
    return upd, bool(ok.value)


def roadmap_updates(map_new, updated, vertex_states, edges, copy_layer_per_edge: bool = False):
    """LazyPRMStarMinUpdateMaintainer's per-vertex / per-edge questions restated against `updated` (the new map's
    layer, [rows, cols]): (vertex_flags [nv] uint8, edge_flags [ne] uint8). Raises ValueError for an edge index >= nv."""
    lib = _load()
    rows, cols = updated.shape
    g = OrcGrid(None, None, rows, cols, float(map_new.res), float(map_new.cx), float(map_new.cy))
    u = np.asfortranarray(updated, dtype=np.float32)
    s = np.ascontiguousarray(vertex_states, dtype=np.float64).reshape(-1, 7)
    e = np.ascontiguousarray(edges, dtype=np.uint32).reshape(-1, 2)
    vf = np.zeros(s.shape[0], np.uint8)
    ef = np.zeros(e.shape[0], np.uint8)
    rc = lib.orc_roadmap_updates(C.byref(g), u.ctypes.data, s.ctypes.data, s.shape[0], e.ctypes.data, e.shape[0],
                                 int(bool(copy_layer_per_edge)), vf.ctypes.data, ef.ctypes.data)
    if rc != 0:
        raise ValueError("edge index >= number of vertices")
    return vf, ef


def line_cells(s, e):
    """grid_map::LineIterator's cells from index s to index e, its loop as written: int32 [nCells, 2]."""
    lib = _load()
    n = lib.orc_line_cells(int(s[0]), int(s[1]), int(e[0]), int(e[1]), None, 0)
    out = np.zeros((n, 2), np.int32)
    lib.orc_line_cells(int(s[0]), int(s[1]), int(e[0]), int(e[1]), out.ctypes.data, n)
    return out
