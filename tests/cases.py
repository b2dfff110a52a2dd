"""Seeded parity cases shared by oracle/make_golden.py (generation with the compiled reference) and the tests."""
from __future__ import annotations

import math

import numpy as np

from art_planner_b200 import synth


def rot12_from_rpy(roll, pitch, yaw):
    """dPose::rotation (row-major 3x4 float32) the way Pose3FromSE3 builds it from a quaternion (utils.h:25-38)."""
    x, y, z, w = [a.astype(np.float32) for a in synth.quat_from_rpy(roll, pitch, yaw)]
    tx, ty, tz = 2 * x, 2 * y, 2 * z
    twx, twy, twz = tx * w, ty * w, tz * w
    txx, txy, txz = tx * x, ty * x, tz * x
    tyy, tyz, tzz = ty * y, tz * y, tz * z
    n = x.shape[0]
    R = np.zeros((n, 12), np.float32)
    R[:, 0] = 1 - (tyy + tzz); R[:, 1] = txy - twz; R[:, 2] = txz + twy
    R[:, 4] = txy + twz; R[:, 5] = 1 - (txx + tzz); R[:, 6] = tyz - twx
    R[:, 8] = txz - twy; R[:, 9] = tyz + twx; R[:, 10] = 1 - (txx + tyy)
    return R


def flat_holes_terrace():
    m = synth.make_flat_map()
    m.elevation_masked[50:60, 50:70] = -np.inf
    m.elevation_masked[100:103, :] = -np.inf
    m.elevation[120:140, 120:140] = 0.25
    m.elevation_masked[120:140, 120:140] = 0.25
    m.desc = "flat 200x200@0.04 + -inf holes + 0.25 m terrace"
    return m


def ramp():
    m = synth.make_flat_map()
    xs, ys = m.cell_xy()
    m.elevation[:] = (0.2 * xs[:, None] + 0.1 * ys[None, :]).astype(np.float32)
    m.elevation_masked[:] = m.elevation
    m.elevation_masked[30:40, 30:40] = -np.inf
    m.desc = "planar ramp 200x200@0.04 (0.2 x + 0.1 y) + -inf hole"
    return m


def c4_map():
    """BASELINE configs[3]: 256x256 crop of the C2 fBm elevation (fp32), same generator, own extent."""
    return synth.make_fbm_map(256, 256, 0.04, seed=2, amp=0.6)


def terraces():
    """Piecewise-constant steps: large coplanar triangle sets, the worst case for the greedy eps-grouping
    (heightfield.cpp:1511-1556)."""
    import dataclasses
    m = synth.make_flat_map()
    e = np.array(m.elevation, dtype=np.float32, order="F")
    r, c = np.indices(e.shape)
    e[:] = (0.07 * ((r // 9) % 4) + 0.05 * ((c // 13) % 3)).astype(np.float32)
    return dataclasses.replace(m, elevation=e, elevation_masked=np.asfortranarray(e.copy()), desc="terraces")


def spikes():
    """Gentle fBm with 1 % isolated 0.4 m spikes: single-vertex contacts and very steep triangles."""
    import dataclasses
    m = synth.make_fbm_map(200, 200, amp=0.2)
    e = np.array(m.elevation, dtype=np.float32, order="F")
    k = np.arange(e.size).reshape(e.shape)
    e[synth.hash_uniform(77, 1, k) < 0.01] += 0.4
    mk = np.array(m.elevation_masked, dtype=np.float32, order="F")
    fin = np.isfinite(mk)
    mk[fin] = e[fin]
    return dataclasses.replace(m, elevation=e, elevation_masked=mk, desc="spikes")


def terraces_tilted():
    """The terraces sheared by a small planar ramp: every terrace is a large set of triangles whose planes are equal only
    up to rounding -- epsilon-grouping near its threshold instead of exactly coplanar."""
    import dataclasses
    m = terraces()
    xs, ys = m.cell_xy()
    e = (m.elevation.astype(np.float64) + 0.013 * xs[:, None] - 0.007 * ys[None, :]).astype(np.float32)
    e = np.asfortranarray(e)
    return dataclasses.replace(m, elevation=e, elevation_masked=e.copy(order="F"), desc="terraces + planar shear")


#: "rough" regime of SURVEY 8(a10) / 8(d): most torso boxes get past the collider's early outs (port statistics on this
#: map with HARD_POSES: above 26 %, vertex 22 %, plane 1 %, fall-through 49 %)
HARD = dict(amp=1.2, wavelength=3.0, persistence=0.7)
HARD_POSES = dict(normal_cells=12)


MAPS = {
    "terraces": terraces,
    "terraces_tilted": terraces_tilted,
    "spikes": spikes,
    "fbm_hard": lambda: synth.make_fbm_map(400, 400, **HARD),
    "flat": lambda: synth.make_flat_map(),
    "flat_holes_terrace": flat_holes_terrace,
    "ramp": ramp,
    "fixture": lambda: synth.make_fixture_map(),
    "fbm_rough": lambda: synth.make_fbm_map(400, 400, amp=0.6),
    "fbm_gentle": lambda: synth.make_fbm_map(400, 400, amp=0.15),
}

PARAMS = {"yaml": synth.PARAMS_YAML, "header": synth.PARAMS_HEADER}

# (name, map, params, pose generator)
POSE_CASES = [
    ("c1_flat_yaml", "flat", "yaml", lambda m: synth.make_flat_poses(m, 10000, seed=1)),
    ("c1_flat_header", "flat", "header", lambda m: synth.make_flat_poses(m, 10000, seed=1)),
    ("holes_yaml", "flat_holes_terrace", "yaml", lambda m: synth.make_flat_poses(m, 10000, seed=21, z_range=0.3)),
    ("ramp_yaml", "ramp", "yaml", lambda m: synth.make_terrain_poses(m, 10000, seed=22)),
    ("ramp_header", "ramp", "header", lambda m: synth.make_terrain_poses(m, 10000, seed=23)),
    ("fixture_yaml", "fixture", "yaml", lambda m: synth.make_terrain_poses(m, 20000, seed=9)),
    ("fixture_header", "fixture", "header", lambda m: synth.make_terrain_poses(m, 20000, seed=9)),
    ("fbm_rough_yaml", "fbm_rough", "yaml", lambda m: synth.make_terrain_poses(m, 20000, seed=3)),
    ("fbm_rough_header", "fbm_rough", "header", lambda m: synth.make_terrain_poses(m, 20000, seed=3)),
    ("fbm_gentle_yaml", "fbm_gentle", "yaml", lambda m: synth.make_terrain_poses(m, 20000, seed=3)),
    ("fbm_tilt_yaml", "fbm_rough", "yaml",
     lambda m: synth.make_terrain_poses(m, 20000, seed=31, z_range=0.4, roll_pert=0.7, pitch_pert=0.7)),
    ("ramp_tilt_header", "ramp", "header",
     lambda m: synth.make_terrain_poses(m, 10000, seed=32, z_range=0.3, roll_pert=0.5, pitch_pert=0.5)),
    # the hard regime: epsilon-grouping worst cases and terrain where most torso boxes reach the triangle / plane pass
    ("terraces_yaml", "terraces", "yaml", lambda m: synth.make_terrain_poses(m, 20000, seed=31)),
    ("terraces_header", "terraces", "header", lambda m: synth.make_terrain_poses(m, 20000, seed=33)),
    ("terraces_low_yaml", "terraces", "yaml",
     lambda m: synth.make_terrain_poses(m, 20000, seed=34, z_range=0.25, roll_pert=0.15, pitch_pert=0.2)),
    ("terraces_tilted_yaml", "terraces_tilted", "yaml", lambda m: synth.make_terrain_poses(m, 20000, seed=35, z_range=0.2)),
    ("spikes_yaml", "spikes", "yaml", lambda m: synth.make_terrain_poses(m, 20000, seed=31)),
    ("spikes_header", "spikes", "header", lambda m: synth.make_terrain_poses(m, 20000, seed=36, z_range=0.2)),
    ("fbm_hard_yaml", "fbm_hard", "yaml", lambda m: synth.make_terrain_poses(m, 20000, seed=3, **HARD_POSES)),
    ("fbm_hard_header", "fbm_hard", "header", lambda m: synth.make_terrain_poses(m, 20000, seed=37, **HARD_POSES)),
    ("fbm_hard_low_yaml", "fbm_hard", "yaml",
     lambda m: synth.make_terrain_poses(m, 20000, seed=38, z_range=0.3, roll_pert=0.3, pitch_pert=0.3, **HARD_POSES)),
]


def box_samples(m, n, seed, which, tilt=0.3, zr=0.3):
    """Adversarial raw box poses: arbitrary tilt, centre near the surface (grazing contacts)."""
    k = np.arange(n)
    lx, ly = m.length
    x = m.cx + (synth.hash_uniform(seed, 11, k) - 0.5) * (lx + 1.0)
    y = m.cy + (synth.hash_uniform(seed, 12, k) - 0.5) * (ly + 1.0)
    i, j = m.index_of(x, y)
    layer = m.elevation if which == 0 else m.elevation_masked
    e = layer[i, j].astype(np.float64)
    e = np.where(np.isfinite(e), e, m.elevation[i, j])
    z = e + (0.15 if which == 0 else 0.0) + (synth.hash_uniform(seed, 13 + which, k) * 2 - 1) * zr
    yaw = (synth.hash_uniform(seed + which, 1, k) * 2 - 1) * math.pi
    roll = (synth.hash_uniform(seed + which, 2, k) * 2 - 1) * tilt
    pitch = (synth.hash_uniform(seed + which, 3, k) * 2 - 1) * tilt
    return np.stack([x, y, z], 1).astype(np.float32), rot12_from_rpy(roll, pitch, yaw)


# (name, map, seed, tilt, zr) -- both boxes of the yaml geometry
BOX_CASES = [
    ("box_flat", "flat", 1, 0.3, 0.3),
    ("box_holes", "flat_holes_terrace", 2, 0.3, 0.3),
    ("box_fixture", "fixture", 3, 0.3, 0.3),
    ("box_ramp", "ramp", 4, 0.3, 0.3),
    ("box_fbm_rough", "fbm_rough", 5, 0.3, 0.3),
    ("box_fbm_tilt", "fbm_rough", 7, 1.2, 0.6),
    ("box_terraces", "terraces", 99, 0.9, 0.35),
    ("box_terraces_tilted", "terraces_tilted", 98, 0.4, 0.3),
    ("box_spikes", "spikes", 99, 0.9, 0.35),
    ("box_fbm_hard", "fbm_hard", 97, 0.5, 0.4),
]
BOX_N = 20000

# Port vs compiled reference on seeds no other case uses and on the adversarial maps, pose and box level (yaml geometry;
# golden: tests/golden/reference_fresh.npz): (name, map, n poses, pose seed, n boxes, box seed, tilt, zr)
FRESH_CASES = [
    ("fresh_fixture", "fixture", 5000, 1234, 5000, 4321, 0.8, 0.4),
    ("fresh_ramp", "ramp", 5000, 1234, 5000, 4321, 0.8, 0.4),
    ("fresh_fbm_rough", "fbm_rough", 5000, 1234, 5000, 4321, 0.8, 0.4),
    ("adversarial_terraces", "terraces", 20000, 31, 20000, 99, 0.9, 0.35),
    ("adversarial_spikes", "spikes", 20000, 31, 20000, 99, 0.9, 0.35),
    ("adversarial_terraces_tilted", "terraces_tilted", 20000, 31, 20000, 99, 0.9, 0.35),
]

# (name, map, params, n_edges, n_steps, seed)
# addValidMilestone connection batches (prm_motion_cost.cpp:341-372): (name, map, params, n, seed, dmin, dmax);
# n_interp = (unsigned)(lateralDistance / 0.5) per edge -> 0..6 interior states here
INTERIOR_CASES = [
    ("interior_fbm_rough_yaml", "fbm_rough", "yaml", 4000, 21, 0.05, 3.4),
    ("interior_fixture_header", "fixture", "header", 3000, 22, 0.05, 2.0),
]

EDGE_CASES = [
    ("edges_fbm_rough_yaml", "fbm_rough", "yaml", 3000, 20, 4),
    ("edges_fixture_header", "fixture", "header", 3000, 7, 5),
    ("edges_fbm_hard_yaml", "fbm_hard", "yaml", 4000, 3, 41),
    ("edges_terraces_yaml", "terraces", "yaml", 4000, 4, 42),
]




# OMPL DiscreteMotionValidator with per-edge validSegmentCount and lastValid: (name, map, params, n, seed, dmin, dmax)
SEGMENT_CASES = [
    ("segments_fbm_rough_yaml", "fbm_rough", "yaml", 3000, 51, 0.05, 2.5),
    ("segments_terraces_header", "terraces", "header", 2000, 52, 0.05, 1.5),
]


def se3_bounds(m, reach_z):
    """RealVectorBounds of the SE3 space as Planner::setMap sets them (planner.cpp:146-156)."""
    lx, ly = m.length
    e = m.elevation[np.isfinite(m.elevation)]
    return ([m.cx - lx, m.cy - ly, float(e.min()) - reach_z / 2], [m.cx + lx, m.cy + ly, float(e.max()) + reach_z / 2])


# processors::Basic (basic.cpp:42-106): (name, map, resolution scale, parameters). res scale 1.25 makes the element sizes
# even numbers (asymmetric anchors); the last case has every safety distance 0 (params.h defaults -> OpenCV's 3x3 box).
def _basic_cases():
    from oracle.basic_oracle import BasicParams
    return [
        ("basic_fbm_rough_yaml", "fbm_rough", 1.0, BasicParams()),
        ("basic_fixture_yaml", "fixture", 1.0, BasicParams()),
        ("basic_terraces_even", "terraces", 1.25, BasicParams(foothold_size=0.2, foothold_margin=0.2)),
        ("basic_fbm_hard_known", "fbm_hard", 1.0, BasicParams(unknown_space_untraversable=False, traversability_thres=0.4)),
        ("basic_fbm_gentle_defaults", "fbm_gentle", 1.0, BasicParams(0.5, True, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0)),
    ]


BASIC_CASES = _basic_cases()
