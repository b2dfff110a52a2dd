"""GPU parity (-m gpu) of map change detection (processors::computeChange, change.cpp:9-51) and the roadmap-reuse
questions of LazyPRMStarMinUpdateMaintainer (lazy_prm_star_min_update.cpp:18-91) against the CPU oracle: bit-identical
layers and flags, host entries == device entries, the C++ mirror, error codes and launch counts."""
import ctypes as C

import numpy as np
import pytest

import cases
import roadmap_cases as rc
from roadmap_cases import RES, grid, seeded_grid
from art_planner_b200 import synth

pytestmark = pytest.mark.gpu

THR = 0.1


@pytest.fixture(scope="module")
def rorc():
    """The map-change / roadmap-update restatement (oracle/roadmap_oracle.c)."""
    from oracle import roadmap_orc
    roadmap_orc.build()
    return roadmap_orc


def _small_cases():
    out = {"identical": (seeded_grid(24, 20, 1), seeded_grid(24, 20, 2))}
    for name, c in (("+x", (3 * RES, 0.0)), ("-x", (-3 * RES, 0.0)), ("+y", (0.0, 3 * RES)), ("-y", (0.0, -3 * RES))):
        out[name] = (seeded_grid(24, 20, 3, *c), seeded_grid(24, 20, 4))
    out["fractional"] = (seeded_grid(16, 12, 5, 2.5 * RES, 0.0), seeded_grid(16, 12, 6))
    out["sizes"] = (seeded_grid(24, 20, 7), seeded_grid(16, 16, 8))
    out["sizes-rev"] = (seeded_grid(16, 16, 8), seeded_grid(24, 20, 7))
    out["disjoint"] = (seeded_grid(16, 16, 9), seeded_grid(16, 16, 9, 6.0, 0.0))
    out["old-centre-outside"] = (seeded_grid(16, 16, 9), seeded_grid(16, 16, 9, 1.2, 0.0))
    thr = np.float32(THR)
    e_new = np.zeros((6, 4), np.float32)
    e_old = np.zeros((6, 4), np.float32)
    e_new[0, 0], e_new[1, 0], e_new[2, 0] = thr, np.nextafter(thr, np.float32(1)), -thr
    e_new[3, 0], e_new[4, 0], e_new[5, 0], e_old[5, 0] = np.nan, np.inf, -np.inf, -np.inf
    t_new, t_old = np.ones((6, 4), np.float32), np.ones((6, 4), np.float32)
    t_new[0, 1], t_old[1, 1], t_new[2, 1] = 0.0, 0.0, 0.5
    out["threshold"] = (grid(6, 4, elevation=e_new, trav=t_new), grid(6, 4, elevation=e_old, trav=t_old))
    return out


SMALL = _small_cases()


@pytest.fixture(scope="module")
def ap():
    import art_planner_b200
    from art_planner_b200 import build
    build.build()
    return art_planner_b200


@pytest.fixture(scope="module")
def chk(ap):
    return ap.StateValidityChecker(cases.PARAMS["yaml"], device=0)


@pytest.fixture(scope="module")
def pair1k():
    new, old = synth.make_map_pair(seed=1, index=0, rows=1000, cols=1000, res=0.04, thr=THR)
    states, edges = synth.make_roadmap(old, 10_000, 50_000, seed=2, max_dist=1.5)
    return new, old, states, edges


@pytest.fixture(scope="module")
def pair4k():
    new, old = synth.make_map_pair(seed=4, index=1, rows=4000, cols=4000, res=0.04, thr=THR, octaves=3)
    states, edges = synth.make_roadmap(old, 100_000, 1_000_000, seed=5, max_dist=1.5)
    return new, old, states, edges


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _torch_layers(m):
    """The map with its two layers as column-major CUDA views ([rows, cols] with strides (1, rows))."""
    import torch
    import types
    f = lambda a: torch.from_numpy(np.ascontiguousarray(np.asarray(a, np.float32).T)).cuda().t()
    return types.SimpleNamespace(elevation=f(m.elevation), traversability_thresholded=f(m.traversability_thresholded),
                                 res=m.res, cx=m.cx, cy=m.cy)


def _cell_centre_states(m, rows_idx, cols_idx):
    rows, cols = m.elevation.shape
    s = np.zeros((len(rows_idx), 7))
    s[:, 0] = m.cx + 0.5 * rows * m.res - (rows_idx + 0.5) * m.res
    s[:, 1] = m.cy + 0.5 * cols * m.res - (cols_idx + 0.5) * m.res
    s[:, 6] = 1.0
    return s


def _check_change(chk, rorc, new, old, probe_cells=None):
    """Host float layer, device float layer and the resident bit layer (read back through vertex queries at cell
    centres) all equal orc_compute_change."""
    import torch
    want, _ = rorc.compute_change(new, old, THR)
    got = chk.computeChange(new, old, THR)
    assert np.array_equal(_bits(got), _bits(want))
    rows, cols = want.shape
    if probe_cells is None:
        ii, jj = np.meshgrid(np.arange(rows), np.arange(cols), indexing="ij")
        ii, jj = ii.ravel(), jj.ravel()
    else:
        ii, jj = probe_cells
    vf, _ = chk.roadmapUpdates(_cell_centre_states(new, ii, jj), np.zeros((0, 2), np.uint32))
    assert np.array_equal(vf, want[ii, jj].astype(np.uint8))
    dn, do = _torch_layers(new), _torch_layers(old)
    got_d = chk.computeChange(dn, do, THR)
    torch.cuda.synchronize()
    assert np.array_equal(_bits(got_d.cpu().numpy()), _bits(want))
    chk.computeChange(dn, do, THR, want_layer=False)          # the bit layer alone
    vf2, _ = chk.roadmapUpdates(_cell_centre_states(new, ii, jj), np.zeros((0, 2), np.uint32))
    assert np.array_equal(vf2, vf)
    return want


@pytest.mark.parametrize("name", sorted(SMALL))
def test_change_layers_match_oracle_small(chk, rorc, name):
    new, old = SMALL[name]
    _check_change(chk, rorc, new, old)


def test_change_layers_match_oracle_1000(chk, rorc, pair1k):
    new, old, _, _ = pair1k
    want = _check_change(chk, rorc, new, old)
    assert 0.05 < want.mean() < 0.95


def test_change_layers_match_oracle_4000(chk, rorc, pair4k):
    new, old, _, _ = pair4k
    rng = np.random.default_rng(3)
    probe = (rng.integers(0, 4000, 1_000_000), rng.integers(0, 4000, 1_000_000))
    _check_change(chk, rorc, new, old, probe)


def _roadmap_parity(chk, rorc, new, old, states, edges):
    import torch
    upd = chk.computeChange(new, old, THR)
    want_v, want_e = rorc.roadmap_updates(new, upd, states, edges)
    vf, ef = chk.roadmapUpdates(states, edges)
    assert np.array_equal(vf, want_v) and np.array_equal(ef, want_e)
    dvf, def_ = chk.roadmapUpdates(torch.from_numpy(states).cuda(), torch.from_numpy(edges.astype(np.int32)).cuda())
    torch.cuda.synchronize()
    chk.pollError()
    assert np.array_equal(dvf.cpu().numpy(), vf) and np.array_equal(def_.cpu().numpy(), ef)
    return vf, ef


def test_roadmap_flags_match_oracle_10k_50k(chk, rorc, pair1k):
    new, old, states, edges = pair1k
    vf, ef = _roadmap_parity(chk, rorc, new, old, states, edges)
    for f in (vf, ef):
        assert set(np.bincount(f, minlength=3).nonzero()[0]) == {0, 1, 2}


def test_roadmap_flags_match_oracle_4000_1e6_edges(chk, rorc, pair4k):
    new, old, states, edges = pair4k
    assert len(edges) == 1_000_000
    _roadmap_parity(chk, rorc, new, old, states, edges)


def test_roadmap_outside_and_cell_boundary_endpoints(chk, rorc):
    """Vertices on cell boundaries and on the map's edges, some outside; edges between all of them."""
    new, old = synth.make_map_pair(seed=6, index=2, rows=200, cols=180, res=0.04, thr=THR)
    rows, cols = new.elevation.shape
    rng = np.random.default_rng(8)
    n = 4000
    i = rng.integers(-3, rows + 4, n)
    j = rng.integers(-3, cols + 4, n)
    s = np.zeros((n, 7))
    s[:, 0] = new.cx + 0.5 * rows * new.res - i * new.res          # exactly on row boundaries (and edges)
    s[:, 1] = new.cy + 0.5 * cols * new.res - j * new.res - (rng.random(n) < 0.5) * 0.5 * new.res
    s[:, 6] = 1.0
    edges = rng.integers(0, n, size=(60_000, 2)).astype(np.uint32)
    vf, ef = _roadmap_parity(chk, rorc, new, old, s, edges)
    assert (vf == 2).any() and (vf != 2).any() and (ef == 2).any() and (ef == 1).any()


def test_host_mirror_resets_what_the_reference_resets(ap, rorc, tmp_path):
    exe = rc.build_roadmap_check(tmp_path)
    new, old = synth.make_map_pair(seed=7, index=3, rows=300, cols=260, res=0.04, thr=THR)
    states, edges = synth.make_roadmap(old, 3000, 12_000, seed=9, margin=0.5)
    rng = np.random.default_rng(10)
    vvalid = (rng.random(len(states)) < 0.7).astype(np.uint32)     # LazyPRM: VALIDITY_TRUE = 1, VALIDITY_UNKNOWN = 0
    evalid = (rng.random(len(edges)) < 0.7).astype(np.uint32)
    upd, vv, ev, removed, at = rc.run_roadmap_check(exe, tmp_path, new, old, THR, states, edges, vvalid, evalid)
    want_upd, _ = rorc.compute_change(new, old, THR)
    assert np.array_equal(_bits(upd), _bits(want_upd))
    vf, ef = rorc.roadmap_updates(new, want_upd, states, edges)
    assert np.array_equal(removed, np.nonzero(vf == 2)[0])          # removeOutdatedVertices
    want_vv = np.where((vf != 2) & (vvalid == 1) & (vf == 1), 0, vvalid)
    want_ev = np.where((evalid == 1) & (ef == 1), 0, evalid)        # edges with flag 2 go with their vertex
    assert np.array_equal(vv, want_vv) and np.array_equal(ev, want_ev)
    assert np.array_equal(at, vf)                                   # getUpdatedAtPosition, 2 = out_of_range
    assert (want_vv != vvalid).any() and (want_ev != evalid).any() and len(removed) > 0


def test_errors_nomap_and_bad_edge_indices(ap):
    import torch
    from art_planner_b200 import capi
    c = ap.StateValidityChecker(cases.PARAMS["yaml"], device=0)
    s = np.zeros((4, 7))
    s[:, 6] = 1.0
    with pytest.raises(capi.ArtpError) as ei:
        c.roadmapUpdates(s, np.array([[0, 1]], np.uint32))
    assert ei.value.code == capi.ARTP_E_NOMAP
    new, old = SMALL["identical"]
    c.computeChange(new, old, THR)
    bad = np.array([[0, 1], [2, 4]], np.uint32)
    with pytest.raises(capi.ArtpError) as ei:
        c.roadmapUpdates(s, bad)
    assert ei.value.code == capi.ARTP_E_INVALID
    vf, ef = c.roadmapUpdates(torch.from_numpy(s).cuda(), torch.from_numpy(bad.astype(np.int32)).cuda())
    torch.cuda.synchronize()
    assert ef.cpu().numpy()[1] == 1                                  # fail closed
    with pytest.raises(capi.ArtpError) as ei:
        c.pollError()
    assert ei.value.code == capi.ARTP_E_INVALID
    c.pollError()                                                    # reported once, then cleared
    c.roadmapUpdates(s, bad[:1])


def test_pose_verdicts_unchanged_and_launch_counts(ap, maps, port_lib, pair1k):
    new, old, states, edges = pair1k
    m = maps("fbm_rough")
    c = ap.StateValidityChecker(cases.PARAMS["yaml"], device=0)
    c.setMap(m)
    c.updateHeightField()
    poses = synth.make_terrain_poses(m, 20000, seed=21)
    before = c.isValidBatch(poses)
    c.computeChange(new, old, THR)
    assert c.stats()["last_launches"] == 1
    c.roadmapUpdates(states, edges)
    st = c.stats()
    assert st["last_launches"] == 1
    c.computeChange(new, old, THR, want_layer=False)
    c.roadmapUpdates(states[:10], edges[:0])
    after = c.isValidBatch(poses)
    assert np.array_equal(before, after)
    o = port_lib.Oracle(cases.PARAMS["yaml"], "port")
    o.set_map(m)
    assert np.array_equal(after, o.check_poses(poses))
