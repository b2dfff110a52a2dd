// artp_roadmap.cuh -- map change detection and roadmap invalidation on the device:
//   processors::computeChange              art_planner/src/map/processors/change.cpp:9-51
//   LazyPRMStarMinUpdateMaintainer         lazy_prm_star_min_update.cpp:18-91 (removeOutdatedVertices' isOutOfBounds,
//                                          invalidateUpdatedGraphComponents' wasUpdated(v) / wasUpdated(e))
//   Map::getUpdatedAtPosition / getUpdatedOnLine   map.h:86-89, map.cpp:44-53
// grid_map_core is not in the reference tree; its index <-> position maps, SubmapGeometry and LineIterator are used in
// the written form DESIGN 4.6 gives (buffer start index (0,0)). The submap geometry is computed on the host
// (artp_capi.cu); the kernels see integer start indices and the overlap size only.
//
// The `updated` layer lives on the device as one bit per cell in grid_map order: cell (i, j) of a rows x cols map is
// bit c & 31 of word c >> 5, c = i + j * rows (125 KB at 1000^2, 2 MB at 4000^2: it stays in L2 for the queries).
#pragma once

#include <cstdint>

namespace artp {

// computeChange over one new-map cell per thread. The overlap is [sn, sn + size) in the new map and [so, so + size) in
// the old one (size = 0 when either submap failed: the layer is all ones).
struct ChangeArgs {
  const float *e_new, *t_new, *e_old, *t_old;   // elevation / traversability_thresholded, column-major
  uint32_t rows_new, rows_old, ncell;           // ncell = rows_new * cols_new
  int sn0, sn1, so0, so1, sx, sy;
  float thr;
  uint32_t* bits;                               // (ncell + 31) / 32 words
  float* upd;                                   // nullable: the float layer, exact 0.0f / 1.0f
};

__global__ void __launch_bounds__(256) change_kernel(const ChangeArgs a) {
  const uint32_t stride = gridDim.x * blockDim.x;
  // base is a multiple of 32 for every warp: lane l of a warp owns bit l of one word
  for (uint32_t base = blockIdx.x * blockDim.x; base < a.ncell; base += stride) {
    const uint32_t c = base + threadIdx.x;
    bool updated = true;                                                    // change.cpp:12 Matrix::Ones
    if (c < a.ncell) {
      const int i = (int)(c % a.rows_new) - a.sn0, j = (int)(c / a.rows_new) - a.sn1;
      if ((unsigned)i < (unsigned)a.sx && (unsigned)j < (unsigned)a.sy) {
        const size_t b = (size_t)(a.so0 + i) + (size_t)(a.so1 + j) * a.rows_old;
        const float hd = __ldg(a.e_new + c) - __ldg(a.e_old + b);          // :33
        const bool height_changed = fabsf(hd) > a.thr;                      // :34 (NaN compares false)
        const bool trav_changed = (__ldg(a.t_old + b) - __ldg(a.t_new + c)) > 0.5f;   // :36-37
        updated = height_changed || trav_changed;                           // :38-40
      }
      if (a.upd) a.upd[c] = updated ? 1.0f : 0.0f;
    }
    const unsigned word = __ballot_sync(0xffffffffu, c < a.ncell && updated);
    if ((threadIdx.x & 31) == 0 && c < a.ncell) a.bits[c >> 5] = word;
  }
}

// Geometry of the map the `updated` bits belong to.
struct RoadmapGeom {
  const uint32_t* bits;
  int rows, cols;
  double res, cx, cy;
};

// grid_map::getIndexFromPosition + checkIfPositionWithinMap, as the sampler uses them (artp_sampler.cuh); an index
// outside the layer (rounding at the far edge) counts as outside. The host uses it for the submap corners (artp_capi.cu),
// the roadmap kernel for the vertices.
__host__ __device__ inline bool grid_index(int rows, int cols, double res, double cx, double cy, double px, double py,
                                           int& row, int& col) {
  const double Lx = rows * res, Ly = cols * res;
  const double tx = -((px - cx) - 0.5 * Lx), ty = -((py - cy) - 0.5 * Ly);
  if (!(tx >= 0.0 && ty >= 0.0 && tx < Lx && ty < Ly)) return false;
  row = (int)(-(((px - 0.5 * Lx) - cx) / res));
  col = (int)(-(((py - 0.5 * Ly) - cy) / res));
  return row >= 0 && col >= 0 && row < rows && col < cols;
}

__device__ __forceinline__ bool updated_bit(const RoadmapGeom& g, int row, int col) {
  const uint32_t c = (uint32_t)row + (uint32_t)col * (uint32_t)g.rows;
  return (__ldg(g.bits + (c >> 5)) >> (c & 31)) & 1u;
}

constexpr uint32_t kRoadmapBadEdge = 4u;   // sticky error word: an edge index >= nv (fail closed: flag 1)

// Vertices: one thread each (isOutOfBounds -> 2, else wasUpdated(v) -> 1). Edges: one warp each. Lanes 0 and 1 place
// source and target; then the warp walks grid_map's LineIterator in closed form -- cell k is
//   major = s_major + k * inc_major,  minor = s_minor + inc_minor * floor((den / 2 + k * add) / den)
// (den = delta_major, add = delta_minor <= den, so the iterator's single subtraction per step keeps its numerator in
// [0, den) and the two agree) -- lanes taking k, k + 32, ... and leaving at the first chunk with an updated cell.
__global__ void __launch_bounds__(256) roadmap_kernel(const RoadmapGeom g, const double* __restrict__ vs, size_t nv,
                                                      const uint32_t* __restrict__ edges, size_t ne,
                                                      uint8_t* __restrict__ vflags, uint8_t* __restrict__ eflags,
                                                      uint32_t* __restrict__ err_word) {
  const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nthreads = (size_t)gridDim.x * blockDim.x;
  for (size_t v = tid; v < nv; v += nthreads) {
    int r, c;
    uint8_t f = 2;                                                          // removeOutdatedVertices (:58-72)
    if (grid_index(g.rows, g.cols, g.res, g.cx, g.cy, __ldg(vs + 7 * v), __ldg(vs + 7 * v + 1), r, c)) f = updated_bit(g, r, c) ? 1 : 0;   // :76-80
    vflags[v] = f;
  }
  const int lane = threadIdx.x & 31;
  for (size_t e = tid >> 5; e < ne; e += nthreads >> 5) {
    int r = 0, c = 0;
    bool inside = false, bad = false;
    if (lane < 2) {                                                         // boost::source / boost::target (:84-91)
      const uint32_t vid = __ldg(edges + 2 * e + lane);
      bad = vid >= nv;
      if (!bad) inside = grid_index(g.rows, g.cols, g.res, g.cx, g.cy, __ldg(vs + 7 * (size_t)vid), __ldg(vs + 7 * (size_t)vid + 1), r, c);
    }
    const unsigned bad_mask = __ballot_sync(0xffffffffu, bad);
    const unsigned in_mask = __ballot_sync(0xffffffffu, inside);
    if (bad_mask) {
      if (lane == 0) { eflags[e] = 1; *(volatile uint32_t*)err_word = kRoadmapBadEdge; }
      continue;
    }
    if ((in_mask & 3u) != 3u) {                                             // removed together with its vertex
      if (lane == 0) eflags[e] = 2;
      continue;
    }
    const int s0 = __shfl_sync(0xffffffffu, r, 0), s1 = __shfl_sync(0xffffffffu, c, 0);
    const int e0 = __shfl_sync(0xffffffffu, r, 1), e1 = __shfl_sync(0xffffffffu, c, 1);
    const int d0 = abs(e0 - s0), d1 = abs(e1 - s1);
    const bool xmaj = d0 >= d1;                                             // LineIterator: x major on ties
    const int den = xmaj ? d0 : d1, add = xmaj ? d1 : d0, n = den + 1;
    const int smaj = xmaj ? s0 : s1, smin = xmaj ? s1 : s0;
    const int imaj = (xmaj ? e0 >= s0 : e1 >= s1) ? 1 : -1, imin = (xmaj ? e1 >= s1 : e0 >= s0) ? 1 : -1;
    const bool narrow = den < 65536;                                        // den/2 + k*add fits 32 bits
    bool hit = false;
    for (int k0 = 0; k0 < n && !hit; k0 += 32) {
      const int k = k0 + lane;
      bool h = false;
      if (k < n) {
        int q = 0;
        if (den) q = narrow ? (int)(((uint32_t)(den >> 1) + (uint32_t)k * (uint32_t)add) / (uint32_t)den)
                            : (int)(((uint64_t)(den >> 1) + (uint64_t)k * (uint64_t)add) / (uint64_t)den);
        const int maj = smaj + k * imaj, mn = smin + imin * q;
        h = xmaj ? updated_bit(g, maj, mn) : updated_bit(g, mn, maj);
      }
      hit = __any_sync(0xffffffffu, h);
    }
    if (lane == 0) eflags[e] = hit ? 1 : 0;
  }
}

}  // namespace artp
