"""Shared inputs of the map-change / roadmap-update tests: small hand-built map pairs, the line closed form, and the
C++ mirror driver (tests/host_cpp/roadmap_check.cpp)."""
import os
import shutil
import struct
import subprocess
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RES = 0.125          # a power of two: every cell boundary below is exact in double


def grid(rows, cols, cx=0.0, cy=0.0, res=RES, elevation=None, trav=None):
    """A map with the two layers computeChange reads (float32, Fortran order)."""
    e = np.zeros((rows, cols), np.float32) if elevation is None else elevation
    t = np.ones((rows, cols), np.float32) if trav is None else trav
    return types.SimpleNamespace(elevation=np.asfortranarray(e, dtype=np.float32),
                                 traversability_thresholded=np.asfortranarray(t, dtype=np.float32),
                                 res=res, cx=cx, cy=cy)


def seeded_grid(rows, cols, seed, cx=0.0, cy=0.0, res=RES):
    """Heights in {0, 0.05, 0.1, 0.2} and traversability in {0, 1}, from seed."""
    rng = np.random.default_rng(seed)
    e = rng.choice(np.array([0.0, 0.05, 0.1, 0.2], np.float32), size=(rows, cols))
    t = (rng.random((rows, cols)) < 0.7).astype(np.float32)
    return grid(rows, cols, cx, cy, res, e, t)


def cellwise_change(new, old, thr):
    """The per-cell rule of change.cpp:33-40 on aligned arrays (float32, NaN compares false)."""
    with np.errstate(invalid="ignore"):
        d = np.abs(new.elevation - old.elevation)
        h = d > np.float32(thr)
        t = (old.traversability_thresholded - new.traversability_thresholded) > np.float32(0.5)
    return (h | t).astype(np.float32)


def sub(m, rs, cs):
    return types.SimpleNamespace(elevation=m.elevation[rs, cs], traversability_thresholded=m.traversability_thresholded[rs, cs])


def line_closed_form(s, e):
    """grid_map::LineIterator's cells in closed form: major = s_major + k*inc, minor = s_minor + inc*floor((den/2 + k*add)/den)."""
    d = np.abs(np.subtract(e, s))
    inc = np.where(np.asarray(e) >= np.asarray(s), 1, -1)
    maj = 0 if d[0] >= d[1] else 1
    mnr = 1 - maj
    den, add = int(d[maj]), int(d[mnr])
    k = np.arange(den + 1, dtype=np.int64)
    q = (den // 2 + k * add) // den if den else np.zeros_like(k)
    out = np.zeros((den + 1, 2), np.int64)
    out[:, maj] = s[maj] + k * inc[maj]
    out[:, mnr] = s[mnr] + inc[mnr] * q
    return out


def build_roadmap_check(outdir):
    """g++ the C++ mirror driver against include/artp_host.hpp and libartp.so; returns the executable's path."""
    from art_planner_b200 import build, capi
    if not os.path.exists(capi.LIB_PATH):
        if shutil.which("nvcc") is None:
            return None
        build.build()
    libdir = os.path.dirname(capi.LIB_PATH)
    exe = os.path.join(str(outdir), "roadmap_check")
    subprocess.run(["g++", "-std=c++14", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "host_cpp", "roadmap_check.cpp"), "-o", exe,
                    "-L", libdir, "-l:libartp.so", f"-Wl,-rpath,{libdir}"], check=True)
    return exe


def run_roadmap_check(exe, tmp, new, old, thr, states, edges, vvalid, evalid):
    """Writes the case, runs roadmap_check, returns (updated, vertex_validity, edge_validity, removed, at_position)."""
    fin, fout = os.path.join(str(tmp), "rm_in.bin"), os.path.join(str(tmp), "rm_out.bin")
    rn, cn = new.elevation.shape
    ro, co = old.elevation.shape
    nv, ne = len(states), len(edges)
    with open(fin, "wb") as f:
        f.write(struct.pack("6i", rn, cn, ro, co, nv, ne))
        f.write(struct.pack("6d", new.res, new.cx, new.cy, old.cx, old.cy, thr))
        for m in (new, old):
            f.write(np.asfortranarray(m.elevation, np.float32).tobytes(order="F"))
            f.write(np.asfortranarray(m.traversability_thresholded, np.float32).tobytes(order="F"))
        f.write(np.ascontiguousarray(states, np.float64).tobytes())
        f.write(np.ascontiguousarray(edges, np.uint32).tobytes())
        f.write(np.ascontiguousarray(vvalid, np.uint32).tobytes())
        f.write(np.ascontiguousarray(evalid, np.uint32).tobytes())
    r = subprocess.run([exe, fin, fout], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    raw = open(fout, "rb").read()
    o = 0
    upd = np.frombuffer(raw, np.float32, rn * cn, o).reshape((rn, cn), order="F"); o += 4 * rn * cn
    vv = np.frombuffer(raw, np.uint32, nv, o); o += 4 * nv
    ev = np.frombuffer(raw, np.uint32, ne, o); o += 4 * ne
    nr = int(np.frombuffer(raw, np.uint64, 1, o)[0]); o += 8
    removed = np.frombuffer(raw, np.uint64, nr, o); o += 8 * nr
    at = np.frombuffer(raw, np.uint8, nv, o)
    return upd, vv, ev, removed, at
