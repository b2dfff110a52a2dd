"""Generate tests/golden/*.npz with the reference's own compiled ODE (oracle/_ref/liborc_ref.so).

Needs the reference's sources (REF of oracle/Makefile):  python oracle/make_golden.py [fresh]
(`fresh` rewrites only tests/golden/reference_fresh.npz.)
Inputs are regenerated from seeds by tests/cases.py; the fixtures hold only the packed result masks plus a
checksum of the inputs (so generator drift is detected) -- a few KB each.
"""
from __future__ import annotations

import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import cases  # noqa: E402
from oracle.orc import Oracle, build  # noqa: E402


def digest(*arrays) -> str:
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def main() -> None:
    build("ref")
    out = {}
    maps = {k: f() for k, f in cases.MAPS.items()}
    for name, mk, pk, gen in cases.POSE_CASES:
        m = maps[mk]
        o = Oracle(cases.PARAMS[pk], "reference")
        o.set_map(m)
        poses = gen(m)
        v = o.check_poses(poses)
        out[name + "/mask"] = np.packbits(v)
        out[name + "/n"] = np.int64(len(v))
        out[name + "/sha"] = np.array(digest(m.elevation, m.elevation_masked, poses))
        print(f"{name}: n={len(v)} valid={int(v.sum())}")
    for name, mk, seed, tilt, zr in cases.BOX_CASES:
        m = maps[mk]
        o = Oracle(cases.PARAMS["yaml"], "reference")
        o.set_map(m)
        for which in (0, 1):
            org, rot = cases.box_samples(m, cases.BOX_N, seed, which, tilt, zr)
            hit = o.box_collide(which, org, rot)
            out[f"{name}/{which}/mask"] = np.packbits(hit)
            out[f"{name}/{which}/sha"] = np.array(digest(m.elevation, m.elevation_masked, org, rot))
            print(f"{name}/{which}: hit={int(hit.sum())}")
    from art_planner_b200 import synth
    for name, mk, pk, n, steps, seed in cases.EDGE_CASES:
        m = maps[mk]
        o = Oracle(cases.PARAMS[pk], "reference")
        o.set_map(m)
        s1, s2 = synth.make_edges(m, n, seed)
        v = o.check_motions(s1, s2, steps)
        c = o.path_length_cost(s1, s2)
        out[name + "/mask"] = np.packbits(v)
        out[name + "/n"] = np.int64(n)
        out[name + "/cost"] = c
        out[name + "/sha"] = np.array(digest(m.elevation, m.elevation_masked, s1, s2))
        print(f"{name}: valid={int(v.sum())}/{n}")
    for name, mk, pk, n, seed, dmin, dmax in cases.INTERIOR_CASES:
        m = maps[mk]
        o = Oracle(cases.PARAMS[pk], "reference")
        o.set_map(m)
        s1, s2 = synth.make_edges(m, n, seed, dmin=dmin, dmax=dmax)
        k = o.check_edge_interiors(s1, s2, None, 0.5)
        out[name + "/prefix"] = k.astype(np.int8)
        out[name + "/sha"] = np.array(digest(m.elevation, m.elevation_masked, s1, s2))
        print(f"{name}: prefix histogram {np.bincount(k).tolist()}")
    for name, mk, pk, n, seed, dmin, dmax in cases.SEGMENT_CASES:
        m = maps[mk]
        o = Oracle(cases.PARAMS[pk], "reference")
        o.set_map(m)
        s1, s2 = synth.make_edges(m, n, seed, dmin=dmin, dmax=dmax)
        low, high = cases.se3_bounds(m, cases.PARAMS[pk].reach_z)
        nd = o.valid_segment_count(low, high, s1, s2)
        v, t = o.check_motions_segments(s1, s2, nd)
        out[name + "/mask"] = np.packbits(v)
        out[name + "/nd"] = nd.astype(np.int32)
        out[name + "/last_t"] = t
        out[name + "/sha"] = np.array(digest(m.elevation, m.elevation_masked, s1, s2))
        print(f"{name}: valid={int(v.sum())}/{n} nd range {nd.min()}..{nd.max()}")
    path = os.path.join(ROOT, "tests", "golden", "reference_masks.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")
    fresh(maps)


def fresh(maps) -> None:
    """tests/golden/reference_fresh.npz: pose and box verdicts of cases.FRESH_CASES."""
    from art_planner_b200 import synth
    out = {}
    for name, mk, n_p, p_seed, n_b, b_seed, tilt, zr in cases.FRESH_CASES:
        m = maps[mk]
        o = Oracle(cases.PARAMS["yaml"], "reference")
        o.set_map(m)
        poses = synth.make_terrain_poses(m, n_p, seed=p_seed)
        v = o.check_poses(poses)
        out[name + "/mask"] = np.packbits(v)
        out[name + "/sha"] = np.array(digest(m.elevation, m.elevation_masked, poses))
        for which in (0, 1):
            org, rot = cases.box_samples(m, n_b, b_seed, which, tilt, zr)
            hit = o.box_collide(which, org, rot)
            out[f"{name}/{which}/mask"] = np.packbits(hit)
            out[f"{name}/{which}/sha"] = np.array(digest(m.elevation, m.elevation_masked, org, rot))
        print(f"{name}: valid={int(v.sum())}/{n_p}")
    path = os.path.join(ROOT, "tests", "golden", "reference_fresh.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    if sys.argv[1:] == ["fresh"]:
        build("ref")
        fresh({k: f() for k, f in cases.MAPS.items()})
    else:
        main()
