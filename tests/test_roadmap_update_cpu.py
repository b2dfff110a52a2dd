"""CPU: the oracle's restatement of processors::computeChange (change.cpp:9-51) and of the roadmap-reuse questions of
LazyPRMStarMinUpdateMaintainer (lazy_prm_star_min_update.cpp:18-91) against hand-worked cases, grid_map's LineIterator
against its closed form, and the C++ mirror (include/artp_host.hpp) compiling and failing loudly without a GPU."""
import subprocess

import numpy as np
import pytest

import roadmap_cases as rc
from roadmap_cases import RES, grid, seeded_grid, cellwise_change, sub

THR = 0.1


@pytest.fixture(scope="module")
def rorc():
    """The map-change / roadmap-update restatement (oracle/roadmap_oracle.c)."""
    from oracle import roadmap_orc
    roadmap_orc.build()
    return roadmap_orc


# ---- LineIterator -------------------------------------------------------------------------------------------------
LINES = {
    "along-y": ((3, 1), (3, 6), [(3, j) for j in range(1, 7)]),
    "along-x": ((1, 3), (6, 3), [(i, 3) for i in range(1, 7)]),
    "diagonal": ((0, 0), (4, 4), [(k, k) for k in range(5)]),
    "tie-x-major": ((0, 0), (3, -3), [(k, -k) for k in range(4)]),          # delta.x == delta.y: x is the major axis
    "shallow+x+y": ((0, 0), (7, 2), [(0, 0), (1, 0), (2, 1), (3, 1), (4, 1), (5, 1), (6, 2), (7, 2)]),
    "shallow-x+y": ((0, 0), (-7, 2), [(0, 0), (-1, 0), (-2, 1), (-3, 1), (-4, 1), (-5, 1), (-6, 2), (-7, 2)]),
    "shallow+x-y": ((0, 0), (7, -2), [(0, 0), (1, 0), (2, -1), (3, -1), (4, -1), (5, -1), (6, -2), (7, -2)]),
    "shallow-x-y": ((0, 0), (-7, -2), [(0, 0), (-1, 0), (-2, -1), (-3, -1), (-4, -1), (-5, -1), (-6, -2), (-7, -2)]),
    "steep+y": ((0, 0), (2, 7), [(0, 0), (0, 1), (1, 2), (1, 3), (1, 4), (1, 5), (2, 6), (2, 7)]),
    "steep-y": ((5, 5), (3, -2), [(5, 5), (5, 4), (4, 3), (4, 2), (4, 1), (4, 0), (3, -1), (3, -2)]),
    "single-cell": ((4, 4), (4, 4), [(4, 4)]),
    "forward": ((0, 0), (4, 1), [(0, 0), (1, 0), (2, 1), (3, 1), (4, 1)]),
    "reversed": ((4, 1), (0, 0), [(4, 1), (3, 1), (2, 0), (1, 0), (0, 0)]),
}


@pytest.mark.parametrize("name", sorted(LINES))
def test_line_iterator_hand_worked(rorc, name):
    s, e, want = LINES[name]
    got = rorc.line_cells(s, e)
    assert got.tolist() == [list(c) for c in want]
    assert np.array_equal(rc.line_closed_form(s, e), got)


def test_line_is_not_symmetric(rorc):
    """Bresenham is not symmetric: the cell set of (0,0) -> (4,1) differs from that of (4,1) -> (0,0)."""
    a = {tuple(c) for c in rorc.line_cells((0, 0), (4, 1))}
    b = {tuple(c) for c in rorc.line_cells((4, 1), (0, 0))}
    assert a != b and (2, 1) in a and (2, 0) in b


def test_line_closed_form_equals_iterative_walk(rorc):
    """The device's closed form equals LineIterator's loop on 10^5 random lines (lengths up to 600 cells)."""
    rng = np.random.default_rng(17)
    n = 100_000
    s = rng.integers(0, 600, size=(n, 2))
    d = rng.integers(-300, 301, size=(n, 2)) * (rng.random((n, 1)) < 0.9) + rng.integers(-3, 4, size=(n, 2))
    e = s + d
    for i in range(n):
        it = rorc.line_cells(s[i], e[i])
        cf = rc.line_closed_form(s[i], e[i])
        assert np.array_equal(it, cf), (s[i], e[i])
        assert tuple(it[0]) == tuple(s[i]) and tuple(it[-1]) == tuple(e[i])


# ---- computeChange ------------------------------------------------------------------------------------------------
def _expect_ones_except(new, region_new, old, region_old, thr=THR):
    want = np.ones(new.elevation.shape, np.float32, order="F")
    want[region_new] = cellwise_change(sub(new, *region_new), sub(old, *region_old), thr)
    return want


def test_change_identical_geometry_is_the_whole_map(rorc):
    new, old = seeded_grid(24, 20, 1), seeded_grid(24, 20, 2)
    upd, ok = rorc.compute_change(new, old, THR)
    assert ok and np.array_equal(upd, cellwise_change(new, old, THR))


@pytest.mark.parametrize("axis,sign", [(0, 1), (0, -1), (1, 1), (1, -1)], ids=["+x", "-x", "+y", "-y"])
def test_change_integer_shift(rorc, axis, sign):
    """The new map is 3 cells further along +-x / +-y. Cell i of the new map lies on cell i -+ 3 of the old one (the row
    index grows towards -x, the column index towards -y)."""
    rows, cols, k = 24, 20, 3
    c = [0.0, 0.0]
    c[axis] = sign * k * RES
    new, old = seeded_grid(rows, cols, 3, *c), seeded_grid(rows, cols, 4)
    full = [slice(None), slice(None)]
    n = (rows, cols)[axis]
    rn, ro = list(full), list(full)
    if sign > 0:
        rn[axis], ro[axis] = slice(k, n), slice(0, n - k)
    else:
        rn[axis], ro[axis] = slice(0, n - k), slice(k, n)
    upd, ok = rorc.compute_change(new, old, THR)
    assert ok and np.array_equal(upd, _expect_ones_except(new, tuple(rn), old, tuple(ro)))


def test_change_fractional_shift(rorc):
    """2.5 cells along +x: the new map's submap starts at row 2 (the old top edge falls mid-cell), the old one at row 0,
    and both are rows - 2 long (getSubmapInformation's inclusive bottom-right index)."""
    rows, cols = 16, 12
    new, old = seeded_grid(rows, cols, 5, 2.5 * RES, 0.0), seeded_grid(rows, cols, 6)
    upd, ok = rorc.compute_change(new, old, THR)
    want = _expect_ones_except(new, (slice(2, rows), slice(None)), old, (slice(0, rows - 2), slice(None)))
    assert ok and np.array_equal(upd, want)


def test_change_different_sizes(rorc):
    """A 24 x 20 new map around a 16 x 16 old one (same centre): the old map is compared with rows 4..19, cols 2..17."""
    new, old = seeded_grid(24, 20, 7), seeded_grid(16, 16, 8)
    upd, ok = rorc.compute_change(new, old, THR)
    assert ok and np.array_equal(upd, _expect_ones_except(new, (slice(4, 20), slice(2, 18)), old, (slice(None), slice(None))))
    # and the other way round: the small new map lies entirely in the old one
    upd2, ok2 = rorc.compute_change(old, new, THR)
    assert ok2 and np.array_equal(upd2, _expect_ones_except(old, (slice(None), slice(None)), new, (slice(4, 20), slice(2, 18))))


@pytest.mark.parametrize("where", ["disjoint", "old-centre-outside"])
def test_change_without_overlap_is_all_ones(rorc, where):
    """Disjoint maps, and maps that overlap while the old centre is outside the new map: a submap fails, all ones."""
    rows, cols = 16, 16
    off = 3.0 * rows * RES if where == "disjoint" else 0.6 * rows * RES
    new, old = seeded_grid(rows, cols, 9), seeded_grid(rows, cols, 9, off, 0.0)
    upd, ok = rorc.compute_change(new, old, THR)
    assert not ok and (upd == 1.0).all()


def test_change_threshold_is_strict_and_only_trav_loss_counts(rorc):
    thr = np.float32(THR)
    e_old = np.zeros((6, 4), np.float32)
    e_new = np.zeros((6, 4), np.float32)
    e_new[0, 0] = thr                                  # exactly at thr: not updated
    e_new[1, 0] = np.nextafter(thr, np.float32(1))     # one ulp above: updated
    e_new[2, 0] = -thr                                 # |difference| == thr: not updated
    e_new[3, 0] = np.nan                               # NaN compares false: not updated
    e_new[4, 0] = np.inf                               # inf: updated
    e_new[5, 0] = -np.inf
    e_old[5, 0] = -np.inf                              # -inf - -inf = NaN: not updated
    t_old = np.ones((6, 4), np.float32)
    t_new = np.ones((6, 4), np.float32)
    t_new[0, 1] = 0.0                                  # 1 -> 0: updated
    t_old[1, 1] = 0.0                                  # 0 -> 1: not updated
    t_new[2, 1] = 0.5                                  # 1 -> 0.5: a drop of exactly 0.5 is not > 0.5
    new, old = grid(6, 4, elevation=e_new, trav=t_new), grid(6, 4, elevation=e_old, trav=t_old)
    upd, ok = rorc.compute_change(new, old, THR)
    want = np.zeros((6, 4), np.float32)
    want[1, 0] = want[4, 0] = want[0, 1] = 1.0
    assert ok and np.array_equal(upd, want)


def test_change_on_the_synthetic_pair(rorc):
    """make_map_pair: the overlap is compared, the rest of the new map is all ones, and every kind of seeded change
    is present (exact-threshold cells not updated, NaN cells not updated)."""
    from art_planner_b200 import synth
    new, old = synth.make_map_pair(seed=3, index=0, rows=300, cols=260, thr=THR)
    upd, ok = rorc.compute_change(new, old, THR)
    assert ok
    assert set(np.unique(upd)) == {0.0, 1.0}
    frac = upd.mean()
    assert 0.1 < frac < 0.9
    again = synth.make_map_pair(seed=3, index=0, rows=300, cols=260, thr=THR)[0]
    assert np.array_equal(again.elevation, new.elevation, equal_nan=True)        # pure function of its arguments
    assert (new.elevation == np.float32(THR)).sum() > 0 and np.isnan(new.elevation).sum() > 0


# ---- roadmap questions ------------------------------------------------------------------------------------------
def _cell_centre(m, i, j):
    rows, cols = m.elevation.shape
    return m.cx + 0.5 * rows * m.res - (i + 0.5) * m.res, m.cy + 0.5 * cols * m.res - (j + 0.5) * m.res


def test_roadmap_hand_worked(rorc):
    """One updated cell (2, 1) in a 10 x 8 map: vertex flags, an edge that crosses it in one direction only, an edge
    with an endpoint outside, an edge between updated / clean vertices."""
    m = grid(10, 8, cx=0.3, cy=-0.2)
    upd = np.zeros((10, 8), np.float32, order="F")
    upd[2, 1] = 1.0
    pts = [_cell_centre(m, 0, 0), _cell_centre(m, 4, 1), _cell_centre(m, 2, 1), (m.cx + 5.0, m.cy), _cell_centre(m, 9, 7)]
    states = np.zeros((len(pts), 7))
    states[:, :2] = pts
    states[:, 6] = 1.0
    edges = np.array([[0, 1], [1, 0], [0, 3], [3, 4], [2, 4], [4, 4]], np.uint32)
    vf, ef = rorc.roadmap_updates(m, upd, states, edges)
    assert vf.tolist() == [0, 0, 1, 2, 0]
    # (0,0) -> (4,1) visits (2,1); (4,1) -> (0,0) visits (2,0) instead
    assert ef.tolist() == [1, 0, 2, 2, 1, 0]
    vf2, ef2 = rorc.roadmap_updates(m, upd, states, edges, copy_layer_per_edge=True)
    assert np.array_equal(vf, vf2) and np.array_equal(ef, ef2)
    with pytest.raises(ValueError):
        rorc.roadmap_updates(m, upd, states, np.array([[0, 5]], np.uint32))


def test_roadmap_map_edges_and_cell_boundaries(rorc):
    """Positions on the map's own edges (the top / left edges are inside, the bottom / right ones are not) and on
    interior cell boundaries (they belong to the cell with the larger index: index = (int)(distance from the top / res))."""
    m = grid(8, 8, cx=0.0, cy=0.0)
    upd = np.zeros((8, 8), np.float32, order="F")
    upd[3, 4] = 1.0
    L = 8 * RES
    pts = [(0.5 * L, 0.0), (-0.5 * L, 0.0), (0.0, 0.5 * L), (0.0, -0.5 * L),    # top, bottom, left, right edge
           (0.5 * L - 3 * RES, 0.5 * L - 4 * RES),                               # the corner of cells (2..3, 3..4)
           (0.5 * L - 3 * RES, 0.5 * L - 4.5 * RES)]
    states = np.zeros((len(pts), 7))
    states[:, :2] = pts
    vf, _ = rorc.roadmap_updates(m, upd, states, np.zeros((0, 2), np.uint32))
    assert vf.tolist() == [0, 2, 0, 2, 1, 1]


def test_host_mirror_compiles_and_fails_loudly_without_gpu(tmp_path):
    import torch
    exe = rc.build_roadmap_check(tmp_path)
    if exe is None:
        pytest.skip("libartp.so not built and nvcc absent")
    r = subprocess.run([exe, "--expect-no-gpu"], capture_output=True, text=True)
    if torch.cuda.is_available():
        assert r.returncode == 3
    else:
        assert r.returncode == 0 and "failed loudly" in r.stdout and "CUDA" in r.stdout
