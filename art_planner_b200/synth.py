"""Deterministic synthetic inputs for the art_planner hot path (SURVEY.md section 8d).

Every generator is a pure function of (seed, index): a counter-based splitmix64 hash feeds all
random draws, so the CPU oracle and the GPU path consume bit-identical arrays and any rank can
regenerate its own shard without communication.

Layer layout follows grid_map (the reference's map container; call sites
art_planner/src/validity_checker/height_map_box_checker.cpp:41-53): a layer is a column-major
rows x cols float32 matrix, cell (i, j) centred at
    x = cx + Lx/2 - (i + 0.5) * res,   y = cy + Ly/2 - (j + 0.5) * res.
`elevation` is finite everywhere; `elevation_masked` equals `elevation` where traversable and -inf
elsewhere (art_planner/src/map/processors/basic.cpp:102-105).
"""
from __future__ import annotations

import dataclasses
import math

import numpy as np

_M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def _splitmix64(x: np.ndarray) -> np.ndarray:
    x = (x + np.uint64(0x9E3779B97F4A7C15)) & _M64
    z = x
    z = ((z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)) & _M64
    z = ((z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)) & _M64
    return z ^ (z >> np.uint64(31))


def hash_u64(seed: int, stream: int, idx) -> np.ndarray:
    """64-bit hash of (seed, stream, idx); idx may be an int array."""
    with np.errstate(over="ignore"):
        idx = np.asarray(idx, dtype=np.uint64)
        k = _splitmix64(np.uint64(seed) * np.uint64(0x632BE59BD9B4E019) + np.uint64(stream))
        return _splitmix64(idx ^ k)


def hash_uniform(seed: int, stream: int, idx) -> np.ndarray:
    """U[0,1) doubles, pure function of (seed, stream, idx)."""
    return (hash_u64(seed, stream, idx) >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


# ---------------------------------------------------------------------------------------------
# robot geometry presets
# ---------------------------------------------------------------------------------------------
@dataclasses.dataclass(frozen=True)
class RobotParams:
    """The fields of art_planner::Params the hot path reads (params.h:14-123)."""
    torso_length: float
    torso_width: float
    torso_height: float
    torso_off_x: float
    torso_off_y: float
    torso_off_z: float
    feet_off_x: float
    feet_off_y: float
    feet_off_z: float
    reach_x: float
    reach_y: float
    reach_z: float
    unknown_space_untraversable: bool = True
    use_directional_cost: bool = True
    max_lon_vel: float = 0.5
    max_lat_vel: float = 0.1
    max_ang_vel: float = 0.5


#: shipped configuration, art_planner_ros/config/params.yaml:55-71 (+ :11, :39-43)
PARAMS_YAML = RobotParams(1.31, 0.65, 0.30, 0.0, 0.0, 0.04, 0.51, 0.20, -0.475, 0.2, 0.2, 0.2,
                          True, True, 0.5, 0.1, 0.5)
#: header defaults, art_planner/include/art_planner/params.h:26,73-76,90-117
PARAMS_HEADER = RobotParams(1.05, 0.55, 0.2, 0.0, 0.0, 0.0, 0.362, 0.225, -0.525, 0.25, 0.1, 0.15,
                            True, False, 0.5, 0.1, 0.5)


# ---------------------------------------------------------------------------------------------
# maps
# ---------------------------------------------------------------------------------------------
@dataclasses.dataclass
class SynthMap:
    elevation: np.ndarray          # float32 [rows, cols], Fortran (column-major) order
    elevation_masked: np.ndarray   # float32 [rows, cols], Fortran order
    res: float
    cx: float
    cy: float
    desc: str
    traversability_thresholded: np.ndarray | None = None   # float32 0 / 1, Fortran order (make_map_pair)

    @property
    def rows(self) -> int:
        return self.elevation.shape[0]

    @property
    def cols(self) -> int:
        return self.elevation.shape[1]

    @property
    def length(self):
        return self.rows * self.res, self.cols * self.res

    def cell_xy(self):
        lx, ly = self.length
        x = self.cx + 0.5 * lx - (np.arange(self.rows) + 0.5) * self.res
        y = self.cy + 0.5 * ly - (np.arange(self.cols) + 0.5) * self.res
        return x, y

    def index_of(self, x, y):
        """grid_map getIndexFromPosition (clamped)."""
        lx, ly = self.length
        i = np.floor((self.cx + 0.5 * lx - x) / self.res).astype(np.int64)
        j = np.floor((self.cy + 0.5 * ly - y) / self.res).astype(np.int64)
        return np.clip(i, 0, self.rows - 1), np.clip(j, 0, self.cols - 1)


_GRAD = np.array([[1, 0], [-1, 0], [0, 1], [0, -1],
                  [0.7071067811865476, 0.7071067811865476], [-0.7071067811865476, 0.7071067811865476],
                  [0.7071067811865476, -0.7071067811865476], [-0.7071067811865476, -0.7071067811865476]])


def _gradient_noise(seed: int, octave: int, u: np.ndarray, v: np.ndarray) -> np.ndarray:
    """Classic 2-D gradient ("Perlin") noise on lattice coords (u, v), gradients hashed per node."""
    u0 = np.floor(u)
    v0 = np.floor(v)
    fu = u - u0
    fv = v - v0
    iu = u0.astype(np.int64)
    iv = v0.astype(np.int64)

    def node(di, dj):
        key = ((iu + di) & 0xFFFFFFFF).astype(np.uint64) << np.uint64(32) | ((iv + dj) & 0xFFFFFFFF).astype(np.uint64)
        g = _GRAD[(hash_u64(seed, 1000 + octave, key) & np.uint64(7)).astype(np.int64)]
        return g[..., 0] * (fu - di) + g[..., 1] * (fv - dj)

    su = fu * fu * fu * (fu * (fu * 6 - 15) + 10)
    sv = fv * fv * fv * (fv * (fv * 6 - 15) + 10)
    n00, n10, n01, n11 = node(0, 0), node(1, 0), node(0, 1), node(1, 1)
    a = n00 + su * (n10 - n00)
    b = n01 + su * (n11 - n01)
    return a + sv * (b - a)


def fbm_height(seed: int, x: np.ndarray, y: np.ndarray, amp: float, wavelength: float = 8.0,
               octaves: int = 5, persistence: float = 0.5) -> np.ndarray:
    """fBm of gradient noise: `octaves` octaves, base wavelength in metres, peak amplitude ~amp; every octave has
    `persistence` times the amplitude of the previous one (0.5 = the classic 1/f spectrum)."""
    h = np.zeros(np.broadcast(x, y).shape, dtype=np.float64)
    a, f, norm = 1.0, 1.0 / wavelength, 0.0
    for o in range(octaves):
        h += a * _gradient_noise(seed, o, x * f + 0.37 * (o + 1), y * f + 0.61 * (o + 1))
        norm += a
        a *= persistence
        f *= 2.0
    return h * (amp * 1.4142135623730951 / norm)


def make_flat_map(rows=200, cols=200, res=0.04, height=0.0, cx=0.0, cy=0.0) -> SynthMap:
    """C1: exactly flat, fully traversable."""
    e = np.full((rows, cols), height, dtype=np.float32, order="F")
    return SynthMap(e, e.copy(order="F"), res, cx, cy, f"flat {rows}x{cols}@{res} h={height}")


def make_fbm_map(rows=1000, cols=1000, res=0.04, seed=2, amp=0.6, wavelength=8.0, octaves=5,
                 blob_frac=0.02, n_walls=6, wall_height=0.5, cx=0.0, cy=0.0, persistence=0.5) -> SynthMap:
    """C2/C5: fBm terrain + a few step walls; ~blob_frac of the cells in 0.3-1 m square blobs are
    untraversable (-inf in `elevation_masked`)."""
    m = SynthMap(np.zeros((rows, cols), np.float32, order="F"), np.zeros((1, 1), np.float32), res, cx, cy, "")
    x, y = m.cell_xy()
    lx, ly = m.length
    e = fbm_height(seed, x[:, None], y[None, :], amp, wavelength, octaves, persistence)
    # step walls: axis-aligned slabs raised by wall_height
    for w in range(n_walls):
        u = hash_uniform(seed, 2000 + w, np.arange(5))
        wx = cx - 0.5 * lx + u[0] * lx
        wy = cy - 0.5 * ly + u[1] * ly
        length = 2.0 + 6.0 * u[2]
        thick = 0.2 + 0.4 * u[3]
        ex, ey = (length, thick) if u[4] < 0.5 else (thick, length)
        ri = np.nonzero(np.abs(x - wx) < 0.5 * ex)[0]          # the slab is a rectangle of rows x columns
        ci = np.nonzero(np.abs(y - wy) < 0.5 * ey)[0]
        if ri.size and ci.size:
            e[ri[0]:ri[-1] + 1, ci[0]:ci[-1] + 1] += wall_height
    e32 = np.asfortranarray(e.astype(np.float32))
    masked = e32.copy(order="F")
    # untraversable square blobs, 0.3-1.0 m (mean area ~0.46 m^2)
    n_blobs = int(round(blob_frac * lx * ly / 0.46))
    if n_blobs > 0:
        k = np.arange(n_blobs)
        bx = cx - 0.5 * lx + hash_uniform(seed, 3001, k) * lx
        by = cy - 0.5 * ly + hash_uniform(seed, 3002, k) * ly
        bs = 0.3 + 0.7 * hash_uniform(seed, 3003, k)
        i0, j1 = m.index_of(bx + 0.5 * bs, by - 0.5 * bs)
        i1, j0 = m.index_of(bx - 0.5 * bs, by + 0.5 * bs)
        for a in range(n_blobs):
            masked[i0[a]:i1[a] + 1, j0[a]:j1[a] + 1] = -np.inf
    desc = (f"fBm gradient noise {rows}x{cols}@{res} seed={seed} amp={amp} wavelength={wavelength} "
            f"octaves={octaves} persistence={persistence} walls={n_walls}x{wall_height}m blobs={blob_frac}")
    return SynthMap(e32, masked, res, cx, cy, desc)


def make_fixture_map(rows=120, cols=120, res=0.05, cx=0.0, cy=0.0) -> SynthMap:
    """The reference's only in-repo synthetic fixture recipe (art_planner/src/ode_test.cpp:24-84),
    regenerated: 6x6 m @0.05, 0.1 m plateau with slots, a 0.8 m wall, one 0.5 m spike; the demo's
    2x2 NaN patch becomes a -inf patch in the masked layer (and stays finite in `elevation`,
    honouring the hot path's input contract: finite or -inf)."""
    e = np.zeros((rows, cols), dtype=np.float32, order="F")
    e[20:60, 20:100] = 0.1
    e[30:34, 20:100] = 0.0
    e[44:46, 20:100] = 0.0
    e[80:84, 10:110] = 0.8
    e[100, 60] = 0.5
    masked = e.copy(order="F")
    masked[10:12, 10:12] = -np.inf
    masked[62:70, 40:52] = -np.inf
    return SynthMap(e, masked, res, cx, cy, f"fixture {rows}x{cols}@{res} (ode_test.cpp recipe)")


# ---------------------------------------------------------------------------------------------
# samples
# ---------------------------------------------------------------------------------------------
def quat_from_rpy(roll, pitch, yaw):
    """setSO3FromRPY, art_planner/include/art_planner/utils.h:100-115. Returns (x, y, z, w)."""
    r2, p2, y2 = roll * 0.5, pitch * 0.5, yaw * 0.5
    cr, cp, cy = np.cos(r2), np.cos(p2), np.cos(y2)
    sr, sp, sy = np.sin(r2), np.sin(p2), np.sin(y2)
    w = cy * cp * cr + sy * sp * sr
    x = cy * cp * sr - sy * sp * cr
    y = sy * cp * sr + cy * sp * cr
    z = sy * cp * cr - cy * sp * sr
    return x, y, z, w


def make_flat_poses(m: SynthMap, n: int, seed: int = 1, start: int = 0, margin: float = 0.25,
                    z_range: float = 0.15) -> np.ndarray:
    """C1 samples: x,y ~ U(-L/2-margin, L/2+margin) (outside-map branches fire), yaw uniform,
    roll = pitch = 0, z = U(-z_range, z_range). Returns [n, 7] float64 (x y z qx qy qz qw)."""
    k = np.arange(start, start + n)
    lx, ly = m.length
    x = m.cx + (hash_uniform(seed, 1, k) - 0.5) * (lx + 2 * margin)
    y = m.cy + (hash_uniform(seed, 2, k) - 0.5) * (ly + 2 * margin)
    z = (hash_uniform(seed, 3, k) * 2 - 1) * z_range
    yaw = (hash_uniform(seed, 4, k) * 2 - 1) * math.pi
    qx, qy, qz, qw = quat_from_rpy(np.zeros(n), np.zeros(n), yaw)
    return np.ascontiguousarray(np.stack([x, y, z, qx, qy, qz, qw], axis=1))


def make_terrain_poses(m: SynthMap, n: int, seed: int = 3, start: int = 0, z_range: float = 0.12,
                       roll_pert: float = math.radians(3.33), pitch_pert: float = math.radians(10.0),
                       xy: tuple | None = None, normal_cells: int = 1) -> np.ndarray:
    """C2/C5 samples: x,y uniform inside the map, yaw uniform, z = cell height + U(+-z_range),
    roll/pitch = terrain-normal aligned + U(+-pert), like SE3FromSE2Sampler::sampleUniform
    (art_planner/src/sampler.cpp:82-131). The normal is the central difference over +-normal_cells cells
    (the reference's estimateNormals averages over estimation_radius = (torso length + width)/4, utils.cpp:213-324;
    normal_cells = 12 is that radius at 0.04 m). Returns [n, 7] float64."""
    k = np.arange(start, start + n)
    lx, ly = m.length
    if xy is None:
        x = m.cx + (hash_uniform(seed, 1, k) - 0.5) * lx * 0.999
        y = m.cy + (hash_uniform(seed, 2, k) - 0.5) * ly * 0.999
    else:
        x, y = xy
    i, j = m.index_of(x, y)
    e = m.elevation
    z = e[i, j].astype(np.float64) + (hash_uniform(seed, 3, k) * 2 - 1) * z_range
    yaw = (hash_uniform(seed, 4, k) * 2 - 1) * math.pi
    # finite-difference normal (x decreases with i, y decreases with j)
    nc = int(normal_cells)
    ip, im = np.clip(i + nc, 0, m.rows - 1), np.clip(i - nc, 0, m.rows - 1)
    jp, jm = np.clip(j + nc, 0, m.cols - 1), np.clip(j - nc, 0, m.cols - 1)
    dzdx = (e[im, j].astype(np.float64) - e[ip, j]) / ((ip - im) * m.res)
    dzdy = (e[i, jm].astype(np.float64) - e[i, jp]) / ((jp - jm) * m.res)
    nrm = np.sqrt(dzdx * dzdx + dzdy * dzdy + 1.0)
    nx, ny, nz = -dzdx / nrm, -dzdy / nrm, 1.0 / nrm
    c, s = np.cos(yaw), np.sin(yaw)
    nbx = c * nx + s * ny
    nby = -s * nx + c * ny
    roll = -np.arctan2(nby, nz) + (hash_uniform(seed, 5, k) * 2 - 1) * roll_pert
    pitch = np.arctan2(nbx, nz) + (hash_uniform(seed, 6, k) * 2 - 1) * pitch_pert
    qx, qy, qz, qw = quat_from_rpy(roll, pitch, yaw)
    return np.ascontiguousarray(np.stack([x, y, z, qx, qy, qz, qw], axis=1))


def make_edges(m: SynthMap, n: int, seed: int = 4, start: int = 0, dmin: float = 0.5, dmax: float = 2.0):
    """C3 edges: s1 as make_terrain_poses, s2 = s1 displaced dmin..dmax m in a random heading with
    its own z / orientation. Returns (s1, s2), each [n, 7] float64."""
    k = np.arange(start, start + n)
    s1 = make_terrain_poses(m, n, seed, start)
    d = dmin + (dmax - dmin) * hash_uniform(seed, 11, k)
    hd = (hash_uniform(seed, 12, k) * 2 - 1) * math.pi
    lx, ly = m.length
    x2 = np.clip(s1[:, 0] + d * np.cos(hd), m.cx - 0.4995 * lx, m.cx + 0.4995 * lx)
    y2 = np.clip(s1[:, 1] + d * np.sin(hd), m.cy - 0.4995 * ly, m.cy + 0.4995 * ly)
    s2 = make_terrain_poses(m, n, seed + 7919, start, xy=(x2, y2))
    return s1, s2


# ---------------------------------------------------------------------------------------------
# sampler inputs: the per-cell layers SE3FromSE2Sampler reads (sampler.cpp:54-131)
# ---------------------------------------------------------------------------------------------
@dataclasses.dataclass
class SamplerLayers:
    """grid_map layers (float32 [rows, cols], Fortran order) the reference's map pre-processing produces
    (processors::Basic normals / plane-fit std-dev, probability_distribution.cpp:20-46 CDFs). Synthetic stand-ins."""
    normal_x: np.ndarray
    normal_y: np.ndarray
    normal_z: np.ndarray
    plane_fit_std_dev: np.ndarray
    sample_probability: np.ndarray
    cum_prob: np.ndarray
    cum_prob_rowwise: np.ndarray        # column 0 of "cum_prob_rowwise_hack", [rows]


def cumulative_distribution(prob: np.ndarray):
    """computeCumulativeProbabilityDistribution (probability_distribution.cpp:20-46) on a float32 matrix: returns
    (cum_prob [rows, cols] Fortran order, cum_prob_rowwise [rows]). Rows without probability mass become NaN rows,
    exactly like the reference's 0/0 division."""
    prob = np.asarray(prob, dtype=np.float32)
    row_sum = prob.sum(axis=1, dtype=np.float32)
    with np.errstate(invalid="ignore", divide="ignore"):
        rowwise = (row_sum / row_sum.sum(dtype=np.float32)).astype(np.float32)
        cum = (prob / row_sum[:, None]).astype(np.float32)
    return np.asfortranarray(np.cumsum(cum, axis=1, dtype=np.float32)), np.cumsum(rowwise, dtype=np.float32)


def make_sampler_layers(m: SynthMap, seed: int = 7, empty_rows: bool = True) -> SamplerLayers:
    """Normals from central differences of the elevation layer, a hashed plane-fit error in [0, 0.8] (so that the
    min(std, 0.5) clamp of sampler.cpp:103 is exercised) and a blocky sample probability with dead regions."""
    e = np.where(np.isfinite(m.elevation), m.elevation, 0.0).astype(np.float64)
    # grid_map axes: row index grows towards -x, column index towards -y
    gx = -np.gradient(e, m.res, axis=0)
    gy = -np.gradient(e, m.res, axis=1)
    nrm = np.sqrt(gx * gx + gy * gy + 1.0)
    rows, cols = m.rows, m.cols
    k = np.arange(rows * cols).reshape(rows, cols)
    std = (0.8 * hash_uniform(seed, 31, k) ** 2).astype(np.float32)
    blk = (np.arange(rows)[:, None] // 16) * 1024 + (np.arange(cols)[None, :] // 16)
    prob = hash_uniform(seed, 32, blk)
    prob = np.where(prob < 0.25, 0.0, prob) * (0.5 + 0.5 * hash_uniform(seed, 33, k))
    if empty_rows:
        prob[rows // 3: rows // 3 + 3, :] = 0.0          # rows without mass -> NaN CDF rows
        prob[0, :] = 0.0
        prob[rows - 1, :] = 0.0
    prob = prob.astype(np.float32)
    cum, cum_row = cumulative_distribution(prob)
    f = lambda a: np.asfortranarray(a.astype(np.float32))
    return SamplerLayers(f(-gx / nrm), f(-gy / nrm), f(1.0 / nrm), np.asfortranarray(std), np.asfortranarray(prob),
                         cum, cum_row)


@dataclasses.dataclass(frozen=True)
class SamplerParams:
    """params.h:79-81 plus the SE3 position bounds Planner::setMap installs (planner.cpp:148-160)."""
    max_roll_pert: float = 3.33 / 180 * math.pi
    max_pitch_pert: float = 10.0 / 180 * math.pi
    sample_from_distribution: bool = True
    low: tuple = (-1.0, -1.0)
    high: tuple = (1.0, 1.0)


def sampler_params_for(m: SynthMap, from_distribution: bool = True) -> SamplerParams:
    lx, ly = m.length
    return SamplerParams(sample_from_distribution=from_distribution, low=(m.cx - lx, m.cy - ly), high=(m.cx + lx, m.cy + ly))


def make_traversability(m: SynthMap, seed: int = 13):
    """Synthetic inputs of processors::Basic: a traversability layer in [0, 1] (smooth noise, low where the terrain is
    steep, a few dead blobs and pin-holes) and an "observed" layer with unobserved patches. float32 F-order."""
    x, y = m.cell_xy()
    e = m.elevation.astype(np.float64)
    gx, gy = np.gradient(e, m.res)
    slope = np.sqrt(gx * gx + gy * gy)
    t = 0.85 - 0.9 * slope + 0.25 * fbm_height(seed, x[:, None], y[None, :], 1.0, wavelength=3.0, octaves=3)
    k = np.arange(e.size).reshape(e.shape)
    t = np.where(hash_uniform(seed, 41, k) < 0.004, 0.0, t)                      # isolated pin-holes
    blk = (np.arange(m.rows)[:, None] // 11) * 4096 + (np.arange(m.cols)[None, :] // 7)
    t = np.where(hash_uniform(seed, 42, blk) < 0.03, 0.05, t)                    # dead blobs
    obs = (hash_uniform(seed, 43, (np.arange(m.rows)[:, None] // 23) * 4096 + (np.arange(m.cols)[None, :] // 29)) > 0.06)
    return (np.asfortranarray(np.clip(t, 0.0, 1.0).astype(np.float32)), np.asfortranarray(obs.astype(np.float32)))


# ---------------------------------------------------------------------------------------------
# map updates: the old / new map pair processors::computeChange compares (change.cpp:9-51) and a roadmap on it
# ---------------------------------------------------------------------------------------------
def _world_map(seed: int, rows: int, cols: int, res: float, cx: float, cy: float, octaves: int) -> SynthMap:
    """A view of the fBm world of `seed` centred at (cx, cy): elevation and a 0 / 1 traversability, both functions of
    the cell centre's world position only, so two views agree wherever their cell centres coincide."""
    m = SynthMap(np.zeros((rows, cols), np.float32, order="F"), np.zeros((1, 1), np.float32), res, cx, cy, "")
    x, y = m.cell_xy()
    e = fbm_height(seed, x[:, None], y[None, :], 0.6, 8.0, octaves).astype(np.float32)
    t = (fbm_height(seed + 1, x[:, None], y[None, :], 1.0, 3.0, 2) > -0.35).astype(np.float32)
    m.elevation = np.asfortranarray(e)
    m.traversability_thresholded = np.asfortranarray(t)
    return m


def _blob_mask(m: SynthMap, bx: float, by: float, half: float):
    """The cells whose centre is within `half` of (bx, by) along both axes, as a (row slice, column slice)."""
    x, y = m.cell_xy()
    ri, ci = np.nonzero(np.abs(x - bx) < half)[0], np.nonzero(np.abs(y - by) < half)[0]
    if not ri.size or not ci.size:
        return slice(0, 0), slice(0, 0)
    return slice(ri[0], ri[-1] + 1), slice(ci[0], ci[-1] + 1)


def make_map_pair(seed: int = 0, index: int = 0, rows: int = 1000, cols: int = 1000, res: float = 0.04,
                  old_rows: int | None = None, old_cols: int | None = None, shift=None, thr: float = 0.1,
                  n_blobs: int = 12, octaves: int = 4):
    """(map_new, map_old) for processors::computeChange: two views of one fBm world, the old one centred at the origin,
    the new one at `shift` (default: a non-integer number of cells, 5-15 % of the map length per axis, drawn from
    (seed, index)), plus seeded changes in the new view -- height blobs above `thr`, below it and exactly at it (flat 0
    in the old view, flat float32(thr) in the new one: |difference| == thr), NaN patches in either view, a -inf patch,
    and traversability switched 1 -> 0 and 0 -> 1. Pure function of its arguments. Layers float32, Fortran order;
    elevation_masked = elevation where traversable and finite, -inf elsewhere."""
    old_rows = rows if old_rows is None else old_rows
    old_cols = cols if old_cols is None else old_cols
    u = hash_uniform(seed, 5000 + 16 * index, np.arange(4))
    if shift is None:
        lx, ly = rows * res, cols * res
        sx = (0.05 + 0.10 * u[0]) * lx * (1 if u[2] < 0.5 else -1)
        sy = (0.05 + 0.10 * u[1]) * ly * (1 if u[3] < 0.5 else -1)
        shift = (sx, sy)
    old = _world_map(seed, old_rows, old_cols, res, 0.0, 0.0, octaves)
    new = _world_map(seed, rows, cols, res, float(shift[0]), float(shift[1]), octaves)
    # blob centres inside the overlap of the two views
    lo_x = max(old.cx - 0.5 * old.length[0], new.cx - 0.5 * new.length[0])
    hi_x = min(old.cx + 0.5 * old.length[0], new.cx + 0.5 * new.length[0])
    lo_y = max(old.cy - 0.5 * old.length[1], new.cy - 0.5 * new.length[1])
    hi_y = min(old.cy + 0.5 * old.length[1], new.cy + 0.5 * new.length[1])
    k = np.arange(8 * n_blobs)
    bx = lo_x + (hi_x - lo_x) * hash_uniform(seed, 5001 + 16 * index, k)
    by = lo_y + (hi_y - lo_y) * hash_uniform(seed, 5002 + 16 * index, k)
    half = 0.1 + 0.4 * hash_uniform(seed, 5003 + 16 * index, k)
    amt = hash_uniform(seed, 5004 + 16 * index, k)
    e_new, e_old = new.elevation, old.elevation
    t_new, t_old = new.traversability_thresholded, old.traversability_thresholded
    thr32 = np.float32(thr)
    for b in range(8 * n_blobs):
        kind = b % 8
        mn, mo = _blob_mask(new, bx[b], by[b], half[b]), _blob_mask(old, bx[b], by[b], half[b])
        if kind == 0:                      # above the threshold
            e_new[mn] += np.float32(thr * (1.05 + 2.0 * amt[b]))
        elif kind == 1:                    # below it
            e_new[mn] += np.float32(thr * 0.9 * amt[b])
        elif kind == 2:                    # exactly at it
            e_old[mo] = 0.0
            e_new[mn] = thr32
        elif kind == 3:                    # NaN in the new view
            e_new[mn] = np.nan
        elif kind == 4:                    # NaN in the old view
            e_old[mo] = np.nan
        elif kind == 5:                    # traversable -> untraversable
            t_old[mo] = 1.0
            t_new[mn] = 0.0
        elif kind == 6:                    # untraversable -> traversable
            t_old[mo] = 0.0
            t_new[mn] = 1.0
        else:                              # -inf (a hole) in the new view
            e_new[mn] = -np.inf if amt[b] < 0.5 else np.inf
    for m in (new, old):
        m.elevation_masked = np.asfortranarray(
            np.where((m.traversability_thresholded > 0.5) & np.isfinite(m.elevation), m.elevation, -np.inf).astype(np.float32))
        m.desc = f"map pair seed={seed} index={index} view {m.rows}x{m.cols}@{res} centre=({m.cx:.4f}, {m.cy:.4f})"
    return new, old


def make_roadmap(m: SynthMap, n_vertices: int, n_edges: int, seed: int = 0, max_dist: float = 1.5, margin: float = 0.0):
    """A PRM-like roadmap: n_vertices SE(3) states uniform over the map's extent grown by `margin` m on every side (so
    some fall outside), and n_edges (source, target) index pairs among the vertex pairs closer than max_dist, found by
    grid binning; which pairs and which direction each edge has are drawn from `seed`. Returns (states [nv, 7] float64,
    edges [ne, 2] uint32); fewer edges when fewer pairs exist."""
    k = np.arange(n_vertices)
    lx, ly = m.length
    x = m.cx - 0.5 * lx - margin + (lx + 2 * margin) * hash_uniform(seed, 6001, k)
    y = m.cy - 0.5 * ly - margin + (ly + 2 * margin) * hash_uniform(seed, 6002, k)
    states = np.zeros((n_vertices, 7), np.float64)
    states[:, 0], states[:, 1], states[:, 6] = x, y, 1.0
    bx = np.floor((x - x.min()) / max_dist).astype(np.int64)
    by = np.floor((y - y.min()) / max_dist).astype(np.int64)
    nbx, nby = int(bx.max()) + 3, int(by.max()) + 3
    bid = (bx + 1) * nby + (by + 1)                     # one empty ring of bins around the occupied ones
    order = np.argsort(bid, kind="stable")
    cnt = np.bincount(bid, minlength=nbx * nby)
    first = np.concatenate([[0], np.cumsum(cnt)[:-1]])
    src_all, dst_all = [], []
    for dx in (-1, 0, 1):
        for dy in (-1, 0, 1):
            nb = bid + dx * nby + dy
            c = cnt[nb]
            src = np.repeat(k, c)
            off = np.arange(int(c.sum())) - np.repeat(np.cumsum(c) - c, c)
            dst = order[np.repeat(first[nb], c) + off]
            keep = src < dst
            src, dst = src[keep], dst[keep]
            d2 = (x[src] - x[dst]) ** 2 + (y[src] - y[dst]) ** 2
            keep = d2 < max_dist * max_dist
            src_all.append(src[keep]); dst_all.append(dst[keep])
    src, dst = np.concatenate(src_all), np.concatenate(dst_all)
    code = src.astype(np.uint64) * np.uint64(n_vertices) + dst.astype(np.uint64)
    pick = np.argsort(hash_u64(seed, 6003, code), kind="stable")[:n_edges]
    src, dst, code = src[pick], dst[pick], code[pick]
    flip = (hash_u64(seed, 6004, code) & np.uint64(1)).astype(bool)
    edges = np.stack([np.where(flip, dst, src), np.where(flip, src, dst)], axis=1).astype(np.uint32)
    return states, np.ascontiguousarray(edges)
