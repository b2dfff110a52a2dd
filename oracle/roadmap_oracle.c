/*
 * oracle/roadmap_oracle.c -- TEST INFRASTRUCTURE ONLY: plain-C restatement of processors::computeChange
 * (art_planner/src/map/processors/change.cpp:9-51) and of the per-vertex / per-edge questions of
 * LazyPRMStarMinUpdateMaintainer (art_planner/src/planners/lazy_prm_star_min_update.cpp:18-91, Map::getUpdatedAtPosition
 * map.h:86-89, Map::getUpdatedOnLine map.cpp:44-53). Built into its own library by oracle/roadmap_orc.py.
 *
 * grid_map_core is not in the reference tree: its getIndexFromPosition / checkIfPositionWithinMap /
 * getPositionFromIndex (restated for the sampler in artp_oracle.c:576-594 and repeated here), boundPositionToRange,
 * getSubmapInformation and LineIterator are restated from their published definitions with buffer start index (0,0).
 * This is the defined, unpinned level the device path shares (DESIGN 4.6); LineIterator's loop is kept as written so
 * that the device's closed form is checked against it.
 *
 * Build: gcc -O2 -ffp-contract=off (no -march, no fast-math), like artp_oracle.c.
 */
#include <float.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct orc_grid {
  const float* elevation;                    /* column-major rows x cols; may be NULL for orc_roadmap_updates */
  const float* traversability_thresholded;
  int rows, cols;
  double res, cx, cy;
} orc_grid;

/* grid_map::getIndexFromPosition (index = (int)(-(position - 0.5*length - mapPosition) / res)) +
 * checkIfPositionWithinMap. Valid iff the position is within the map AND the index is in range (an index one past the
 * end, from rounding, is treated as outside; grid_map would read past the layer there). */
static int gm_grid_index(const orc_grid* g, double px, double py, int* row, int* col) {
  const double Lx = g->rows * g->res, Ly = g->cols * g->res;
  const double vx = ((px - 0.5 * Lx) - g->cx) / g->res, vy = ((py - 0.5 * Ly) - g->cy) / g->res;
  const double tx = -((px - g->cx) - 0.5 * Lx), ty = -((py - g->cy) - 0.5 * Ly);
  if (!(tx >= 0.0 && ty >= 0.0 && tx < Lx && ty < Ly)) return 0;
  *row = (int)(-vx);
  *col = (int)(-vy);
  return *row >= 0 && *col >= 0 && *row < g->rows && *col < g->cols;
}

/* grid_map::getPositionFromIndex (GridMapMath.cpp): position = mapPosition + (0.5*length - 0.5*res) + res * (-index),
 * as artp_oracle.c's gm_position_of_index restates it for the sampler. */
static void gm_grid_position(const orc_grid* g, int row, int col, double pos[2]) {
  const double offx = 0.5 * (g->rows * g->res) - 0.5 * g->res, offy = 0.5 * (g->cols * g->res) - 0.5 * g->res;
  pos[0] = (g->cx + offx) + g->res * (-(double)row);
  pos[1] = (g->cy + offy) + g->res * (-(double)col);
}

/* grid_map::boundPositionToRange: shift into [0, length) relative to the corner, epsilon = 10 * DBL_EPSILON (times |p|
 * when |p| > 1). Eigen evaluates `position - mapPosition + vectorToOrigin` and back left to right per coordinate. */
static void gm_bound_position(double* p, double L, double c) {
  const double vto = 0.5 * L;
  double s = (*p - c) + vto;
  double eps = 10.0 * DBL_EPSILON;
  if (fabs(*p) > 1.0) eps *= fabs(*p);
  if (s <= 0.0) s = eps;
  else if (s >= L) s = L - eps;
  *p = (s + c) - vto;
}

/* grid_map::SubmapGeometry(map, position, length) = getSubmapInformation: returns 1 on success with the submap's start
 * index and size. A corner index outside the map (possible only through rounding) is a failure. */
static int gm_submap(const orc_grid* g, double req_x, double req_y, double req_lx, double req_ly, int start[2], int size[2]) {
  const double Lx = g->rows * g->res, Ly = g->cols * g->res;
  /* corners: topLeft = requested - transform * 0.5 * length with transform = -I (map frame -> buffer order) */
  double tl[2] = {req_x + 0.5 * req_lx, req_y + 0.5 * req_ly};
  double br[2] = {req_x - 0.5 * req_lx, req_y - 0.5 * req_ly};
  gm_bound_position(&tl[0], Lx, g->cx); gm_bound_position(&tl[1], Ly, g->cy);
  gm_bound_position(&br[0], Lx, g->cx); gm_bound_position(&br[1], Ly, g->cy);
  int ti, tj, bi, bj;
  if (!gm_grid_index(g, tl[0], tl[1], &ti, &tj)) return 0;
  if (!gm_grid_index(g, br[0], br[1], &bi, &bj)) return 0;
  /* getPositionFromIndex(topLeft) + 0.5 res = the submap's top-left corner */
  double corner[2];
  gm_grid_position(g, ti, tj, corner);
  corner[0] = corner[0] + 0.5 * g->res;
  corner[1] = corner[1] + 0.5 * g->res;
  size[0] = bi - ti + 1;
  size[1] = bj - tj + 1;
  start[0] = ti; start[1] = tj;
  const double slx = size[0] * g->res, sly = size[1] * g->res;
  const double spx = corner[0] - 0.5 * slx, spy = corner[1] - 0.5 * sly;
  /* getIndexFromPosition(requestedIndexInSubmap, requestedPosition, submapLength, submapPosition): within-map test */
  const double tx = -((req_x - spx) - 0.5 * slx), ty = -((req_y - spy) - 0.5 * sly);
  return tx >= 0.0 && ty >= 0.0 && tx < slx && ty < sly;
}

int orc_compute_change(const orc_grid* mn, const orc_grid* mo, float thr, float* updated, int* overlap_ok) {
  const size_t ncell = (size_t)mn->rows * mn->cols;
  for (size_t c = 0; c < ncell; ++c) updated[c] = 1.0f;                      /* :12 Matrix::Ones */
  int sn[2], zn[2], so[2], zo[2];
  const int ok_new = gm_submap(mn, mo->cx, mo->cy, mo->rows * mo->res, mo->cols * mo->res, sn, zn);   /* :15-18 */
  const int ok_old = gm_submap(mo, mn->cx, mn->cy, mn->rows * mn->res, mn->cols * mn->res, so, zo);   /* :19-22 */
  if (overlap_ok) *overlap_ok = ok_new && ok_old;
  if (!(ok_new && ok_old)) return 0;                                          /* :27 */
  const int sx = zn[0] > zo[0] ? zo[0] : zn[0], sy = zn[1] > zo[1] ? zo[1] : zn[1];   /* :23-25 */
  for (int i = 0; i < sx; ++i) {
    for (int j = 0; j < sy; ++j) {
      const size_t a = (size_t)(sn[0] + i) + (size_t)(sn[1] + j) * mn->rows;
      const size_t b = (size_t)(so[0] + i) + (size_t)(so[1] + j) * mo->rows;
      const float hd = mn->elevation[a] - mo->elevation[b];                   /* :33 */
      const int height_changed = fabsf(hd) > thr;                            /* :34 */
      const int trav_changed = (mo->traversability_thresholded[b] - mn->traversability_thresholded[a]) > 0.5f;   /* :36-37 */
      if (!height_changed && !trav_changed) updated[a] = 0.0f;               /* :38-40 */
    }
  }
  return 0;
}

/* grid_map::LineIterator (initializeIterationParameters + operator++), start index (0,0): Bresenham from s to e. */
typedef struct gm_line { int idx[2], inc1[2], inc2[2], num, den, add, n, k; } gm_line;
static void gm_line_init(gm_line* L, int s0, int s1, int e0, int e1) {
  const int dx = abs(e0 - s0), dy = abs(e1 - s1);
  L->idx[0] = s0; L->idx[1] = s1; L->k = 0;
  L->inc1[0] = L->inc2[0] = e0 >= s0 ? 1 : -1;
  L->inc1[1] = L->inc2[1] = e1 >= s1 ? 1 : -1;
  if (dx >= dy) {                 /* at least one x-value for every y-value */
    L->inc1[0] = 0; L->inc2[1] = 0;
    L->den = dx; L->num = dx / 2; L->add = dy; L->n = dx + 1;
  } else {
    L->inc2[0] = 0; L->inc1[1] = 0;
    L->den = dy; L->num = dy / 2; L->add = dx; L->n = dy + 1;
  }
}
static void gm_line_next(gm_line* L) {
  L->num += L->add;
  if (L->num >= L->den) {
    L->num -= L->den;
    L->idx[0] += L->inc1[0]; L->idx[1] += L->inc1[1];
  }
  L->idx[0] += L->inc2[0]; L->idx[1] += L->inc2[1];
  ++L->k;
}

int orc_line_cells(int s0, int s1, int e0, int e1, int32_t* cells, int cap) {
  gm_line L;
  gm_line_init(&L, s0, s1, e0, e1);
  for (; L.k < L.n; gm_line_next(&L))
    if (L.k < cap) { cells[2 * L.k] = L.idx[0]; cells[2 * L.k + 1] = L.idx[1]; }
  return L.n;
}

int orc_roadmap_updates(const orc_grid* g, const float* updated, const double* vs, size_t nv, const uint32_t* edges,
                        size_t ne, int copy_layer_per_edge, uint8_t* vflags, uint8_t* eflags) {
  for (size_t e = 0; e < 2 * ne; ++e)
    if (edges[e] >= nv) return 1;
  const size_t ncell = (size_t)g->rows * g->cols;
  int* cell = (int*)malloc(sizeof(int) * 2 * (nv ? nv : 1));
  for (size_t v = 0; v < nv; ++v) {
    int r, c;
    /* isOutOfBounds (:94-98) -> removeOutdatedVertices (:58-72); wasUpdated(v) (:76-80, map.h:86-89) */
    if (!gm_grid_index(g, vs[7 * v], vs[7 * v + 1], &r, &c)) { vflags[v] = 2; cell[2 * v] = -1; continue; }
    cell[2 * v] = r; cell[2 * v + 1] = c;
    vflags[v] = updated[(size_t)r + (size_t)c * g->rows] > FLT_EPSILON ? 1 : 0;
  }
  for (size_t e = 0; e < ne; ++e) {
    const uint32_t a = edges[2 * e], b = edges[2 * e + 1];   /* boost::source, boost::target (:84-91) */
    if (cell[2 * a] < 0 || cell[2 * b] < 0) { eflags[e] = 2; continue; }   /* removed with its vertex */
    const float* layer = updated;
    float* copy = NULL;
    if (copy_layer_per_edge) {                 /* map.cpp:46: grid_map::Matrix by value */
      copy = (float*)malloc(sizeof(float) * ncell);
      memcpy(copy, updated, sizeof(float) * ncell);
      layer = copy;
    }
    gm_line L;                                 /* map.cpp:47-51 */
    gm_line_init(&L, cell[2 * a], cell[2 * a + 1], cell[2 * b], cell[2 * b + 1]);
    uint8_t hit = 0;
    for (; L.k < L.n; gm_line_next(&L))
      if (layer[(size_t)L.idx[0] + (size_t)L.idx[1] * g->rows] > FLT_EPSILON) { hit = 1; break; }
    eflags[e] = hit;
    free(copy);
  }
  free(cell);
  return 0;
}

/* Exported (ctypes, oracle/roadmap_orc.py):
 *   orc_compute_change(map_new, map_old, thr, updated, overlap_ok)   updated: rows_new x cols_new floats, column-major;
 *                                                                      *overlap_ok (nullable) = both submaps valid
 *   orc_roadmap_updates(geom, updated, states, nv, edges, ne, copy_layer_per_edge, vertex_flags, edge_flags)
 *       vertex_flags 0 keep, 1 updated, 2 outside; edge_flags 0, 1 updated, 2 an endpoint outside. copy_layer_per_edge
 *       != 0 copies the whole layer for every edge query like `const auto updated = map_->get("updated")`.
 *       Returns 1 if an edge index is >= nv.
 *   orc_line_cells(s0, s1, e0, e1, cells, cap)   LineIterator's cells (up to cap, 2 ints each); returns nCells. */
