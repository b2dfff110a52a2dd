"""CPU-only: the oracle restatement (oracle/artp_oracle.c) against the golden masks produced by the reference's
own compiled ODE (oracle/make_golden.py)."""
import hashlib
import os

import numpy as np
import pytest

import cases
from art_planner_b200 import synth


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def unpack(golden, key, n):
    return np.unpackbits(golden[key])[:n]


@pytest.mark.parametrize("case", cases.POSE_CASES, ids=[c[0] for c in cases.POSE_CASES])
def test_port_pose_masks_match_reference_golden(case, golden, maps, port_lib):
    name, mk, pk, gen = case
    m = maps(mk)
    poses = gen(m)
    assert digest(m.elevation, m.elevation_masked, poses) == str(golden[name + "/sha"]), "generator drift"
    o = port_lib.Oracle(cases.PARAMS[pk], "port")
    o.set_map(m)
    v = o.check_poses(poses)
    ref = unpack(golden, name + "/mask", len(v))
    assert np.array_equal(v, ref)
    # the multi-threaded variant must agree too
    assert np.array_equal(o.check_poses_mt(poses, 4), ref)


@pytest.mark.parametrize("case", cases.BOX_CASES, ids=[c[0] for c in cases.BOX_CASES])
def test_port_box_hits_match_reference_golden(case, golden, maps, port_lib):
    name, mk, seed, tilt, zr = case
    m = maps(mk)
    o = port_lib.Oracle(cases.PARAMS["yaml"], "port")
    o.set_map(m)
    for which in (0, 1):
        org, rot = cases.box_samples(m, cases.BOX_N, seed, which, tilt, zr)
        assert digest(m.elevation, m.elevation_masked, org, rot) == str(golden[f"{name}/{which}/sha"])
        hit = o.box_collide(which, org, rot)
        assert np.array_equal(hit, unpack(golden, f"{name}/{which}/mask", len(hit)))


@pytest.mark.parametrize("case", cases.EDGE_CASES, ids=[c[0] for c in cases.EDGE_CASES])
def test_port_edges_match_reference_golden(case, golden, maps, port_lib):
    name, mk, pk, n, steps, seed = case
    m = maps(mk)
    o = port_lib.Oracle(cases.PARAMS[pk], "port")
    o.set_map(m)
    s1, s2 = synth.make_edges(m, n, seed)
    assert digest(m.elevation, m.elevation_masked, s1, s2) == str(golden[name + "/sha"])
    assert np.array_equal(o.check_motions(s1, s2, steps), unpack(golden, name + "/mask", n))
    assert np.array_equal(o.path_length_cost(s1, s2), golden[name + "/cost"])


@pytest.mark.parametrize("case", cases.INTERIOR_CASES, ids=[c[0] for c in cases.INTERIOR_CASES])
def test_port_edge_interiors_match_reference_golden(case, golden, maps, port_lib):
    name, mk, pk, n, seed, dmin, dmax = case
    m = maps(mk)
    o = port_lib.Oracle(cases.PARAMS[pk], "port")
    o.set_map(m)
    s1, s2 = synth.make_edges(m, n, seed, dmin=dmin, dmax=dmax)
    assert digest(m.elevation, m.elevation_masked, s1, s2) == str(golden[name + "/sha"])
    ref = golden[name + "/prefix"].astype(np.int32)
    assert np.array_equal(o.check_edge_interiors(s1, s2, None, 0.5), ref)
    # explicit counts give the same answer, and the prefix is consistent with per-state validity
    d = np.sqrt((s2[:, 0] - s1[:, 0]) ** 2 + (s2[:, 1] - s1[:, 1]) ** 2)
    ni = (d / 0.5).astype(np.int32)
    assert np.array_equal(o.check_edge_interiors(s1, s2, ni, 0.5), ref)
    assert (ref <= ni).all() and (ref < ni).any() and (ref == ni).any()


def test_edge_with_zero_steps_is_endpoint_check(maps, port_lib):
    m = maps("fixture")
    o = port_lib.Oracle(cases.PARAMS["yaml"], "port")
    o.set_map(m)
    s1, s2 = synth.make_edges(m, 500, 77)
    assert np.array_equal(o.check_motions(s1, s2, 0), o.check_poses(s2))


def test_empty_batches(maps, port_lib):
    m = maps("flat")
    o = port_lib.Oracle(cases.PARAMS["yaml"], "port")
    o.set_map(m)
    assert o.check_poses(np.zeros((0, 7))).shape == (0,)


@pytest.fixture(scope="module")
def fresh():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_fresh.npz"))


def port_equals_compiled_reference(case, maps, port_lib, fresh):
    """Port pose and box verdicts == the compiled reference ODE's (stored by oracle/make_golden.py); returns the
    pose verdicts."""
    name, mk, n_p, p_seed, n_b, b_seed, tilt, zr = case
    m = maps(mk)
    P = port_lib.Oracle(cases.PARAMS["yaml"], "port")
    P.set_map(m)
    poses = synth.make_terrain_poses(m, n_p, seed=p_seed)
    assert digest(m.elevation, m.elevation_masked, poses) == str(fresh[name + "/sha"]), "generator drift"
    a = P.check_poses(poses)
    assert np.array_equal(a, unpack(fresh, name + "/mask", n_p))
    for which in (0, 1):
        org, rot = cases.box_samples(m, n_b, b_seed, which, tilt, zr)
        assert digest(m.elevation, m.elevation_masked, org, rot) == str(fresh[f"{name}/{which}/sha"])
        assert np.array_equal(P.box_collide(which, org, rot), unpack(fresh, f"{name}/{which}/mask", n_b))
    return a


def test_port_equals_compiled_reference_on_fresh_seeds(maps, port_lib, fresh):
    """Fresh seeds (not in reference_masks.npz): port == compiled reference ODE, pose and box level."""
    for case in cases.FRESH_CASES:
        if case[0].startswith("fresh_"):
            port_equals_compiled_reference(case, maps, port_lib, fresh)


@pytest.mark.parametrize("mk", ["terraces", "spikes", "terraces_tilted"])
def test_port_equals_compiled_reference_on_adversarial_maps(mk, maps, port_lib, fresh):
    case = next(c for c in cases.FRESH_CASES if c[0] == "adversarial_" + mk)
    a = port_equals_compiled_reference(case, maps, port_lib, fresh)
    assert 0 < a.sum() < len(a)


def test_hard_regime_exit_mix(maps, port_lib):
    """The 'fbm_hard' map really is the hard regime (SURVEY 8(a10) 'rough'): most torso boxes get past the early outs."""
    import ctypes as C
    m = maps("fbm_hard")
    o = port_lib.Oracle(cases.PARAMS["yaml"], "port")
    o.set_map(m)
    poses = synth.make_terrain_poses(m, 4000, seed=3, **cases.HARD_POSES)
    n = len(poses)
    st = np.zeros(5 * n, np.uint8); hit = np.zeros(5 * n, np.uint8); zv = np.zeros(5 * n, np.uint32)
    f = o.lib.orc_port_pose_box_stats
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]
    assert f(o.h, poses.ctypes.data, n, st.ctypes.data, hit.ctypes.data, zv.ctypes.data) == 0
    torso = np.bincount(st.reshape(n, 5)[:, 0], minlength=8)[:8] / n     # ORC_ST_*: 5 vertex, 6 plane, 7 fall-through
    assert torso[5] + torso[6] + torso[7] >= 0.5 and torso[7] >= 0.4, torso


@pytest.mark.parametrize("case", cases.SEGMENT_CASES, ids=[c[0] for c in cases.SEGMENT_CASES])
def test_port_motion_segments_match_reference_golden(case, golden, maps, port_lib):
    """Per-edge validSegmentCount + DiscreteMotionValidator::checkMotion(s1, s2, lastValid): port == compiled reference."""
    name, mk, pk, n, seed, dmin, dmax = case
    m = maps(mk)
    o = port_lib.Oracle(cases.PARAMS[pk], "port")
    o.set_map(m)
    s1, s2 = synth.make_edges(m, n, seed, dmin=dmin, dmax=dmax)
    assert digest(m.elevation, m.elevation_masked, s1, s2) == str(golden[name + "/sha"])
    low, high = cases.se3_bounds(m, cases.PARAMS[pk].reach_z)
    nd = o.valid_segment_count(low, high, s1, s2)
    assert np.array_equal(nd, golden[name + "/nd"])
    v, t = o.check_motions_segments(s1, s2, nd)
    assert np.array_equal(v, unpack(golden, name + "/mask", n)) and np.array_equal(t, golden[name + "/last_t"])
    # the 2-argument checkMotion (fixed segment count) is the same predicate
    k = 9
    vk, _ = o.check_motions_segments(s1, s2, np.full(n, k, np.int32))
    assert np.array_equal(vk, o.check_motions(s1, s2, k - 1))
