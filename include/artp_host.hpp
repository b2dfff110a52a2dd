// include/artp_host.hpp -- C++ host side of the B200-native art_planner hot path, above the C ABI (artp.h).
//
// Header-only mirror of the reference's plugin classes for this path -- same class and method names, argument meaning
// and error behaviour -- so that art_planner's planners and facade keep calling what they call today:
//   art_planner::StateValidityChecker   include/art_planner/validity_checker/validity_checker.h:21-39
//   ompl::base::MotionValidator         (OMPL DiscreteMotionValidator; call sites prm_motion_cost.cpp:652,
//                                        lazy_prm_star_min_update.cpp:725)
//   art_planner::PathLengthObjective    include/art_planner/objectives/path_length_objective.h, .cpp:26-70
//   art_planner::MotionCostObjective    include/art_planner/objectives/motion_cost_objective.h:19-78, .cpp:28-95
//   processors::computeChange           src/map/processors/change.cpp:9-51 (+ Map::getUpdatedAtPosition, map.h:86-89)
//   LazyPRMStarMinUpdateMaintainer      src/planners/lazy_prm_star_min_update.cpp:18-91, 123-135 (flags only; the Boost
//                                        graph surgery stays with the planner)
// OMPL / Eigen / grid_map are not available in this build image, so the classes are written against three tiny
// stand-ins (State = the seven doubles utils.h:25-38 reads from an SE3StateSpace::StateType, Map = two column-major
// float layers + geometry as grid_map stores them, EdgeMatrix = row-major float matrix). With -DARTP_WITH_OMPL the
// OMPL adapters at the bottom derive from the real ompl::base classes and forward to the same objects.
// There is no CPU fallback: construction throws std::runtime_error if the CUDA library cannot create a handle.
#pragma once

#include <cmath>
#include <cstdint>
#include <functional>
#include <limits>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "artp.h"

namespace artp_host {

// art_planner::Params, the fields this path reads, with the reference's nesting (params.h:14-123).
struct Params {
  struct {
    bool unknown_space_untraversable{true};
    struct {
      float max_query_edge_length{0.5f};
      float risk_threshold{0.1f};
      struct { float energy{0.0f}; float time{1.0f}; float risk{5.0f}; } cost_weights;
    } prm_motion_cost;
  } planner;
  struct {
    struct { bool use_directional_cost{false}; double max_lon_vel{0.5}; double max_lat_vel{0.1}; double max_ang_vel{0.5}; } custom_path_length;
  } objectives;
  struct {
    struct { double length{1.05}; double width{0.55}; double height{0.2}; struct { double x{0}, y{0}, z{0}; } offset; } torso;
    struct { struct { double x{0.362}, y{0.225}, z{-0.525}; } offset; struct { double x{0.25}, y{0.1}, z{0.15}; } reach; } feet;
  } robot;
  struct {
    double max_pitch_pert{10.0 / 180 * 3.14159265358979323846};   // params.h:79
    double max_roll_pert{3.33 / 180 * 3.14159265358979323846};    // params.h:80
    bool sample_from_distribution{true};                            // params.h:81
  } sampler;
  int device{0};   // not in the reference: CUDA device ordinal
};
using ParamsConstPtr = std::shared_ptr<const Params>;

// The SE3StateSpace::StateType fields the reference reads (utils.h:25-38): position + quaternion, doubles.
struct State { double x{0}, y{0}, z{0}, qx{0}, qy{0}, qz{0}, qw{1}; };

// Stand-in for art_planner::Map / grid_map::GridMap: layers are column-major rows x cols (index (i,j) at i + j*rows).
struct Map {
  int rows{0}, cols{0};
  double resolution{0}, position_x{0}, position_y{0};
  std::vector<float> elevation, elevation_masked;
  // layers the sampler reads (Map::getNormal / getPlaneFitStdDev map.h:94-116, probability_distribution.cpp:20-46);
  // cum_prob_rowwise = column 0 of "cum_prob_rowwise_hack". Empty when no sampler is used.
  std::vector<float> normal_x, normal_y, normal_z, plane_fit_std_dev, cum_prob, cum_prob_rowwise;
  // processors::Basic's "traversability_thresholded" (0 / 1) and computeChange's "updated" (change.cpp:50).
  std::vector<float> traversability_thresholded, updated;

  // grid_map getIndexFromPosition + checkIfPositionWithinMap (buffer start index (0,0)); false outside the map (an index
  // past the last cell from rounding counts as outside, DESIGN 4.6).
  bool getIndex(double x, double y, int* row, int* col) const {
    const double lx = rows * resolution, ly = cols * resolution;
    const double tx = -((x - position_x) - 0.5 * lx), ty = -((y - position_y) - 0.5 * ly);
    if (!(tx >= 0.0 && ty >= 0.0 && tx < lx && ty < ly)) return false;
    *row = static_cast<int>(-(((x - 0.5 * lx) - position_x) / resolution));
    *col = static_cast<int>(-(((y - 0.5 * ly) - position_y) / resolution));
    return *row >= 0 && *col >= 0 && *row < rows && *col < cols;
  }
  bool isInside(double x, double y) const { int r, c; return getIndex(x, y, &r, &c); }
  // Map::getUpdatedAtPosition (map.h:86-89): throws std::out_of_range outside the map, as GridMap::atPosition does.
  bool getUpdatedAtPosition(double x, double y) const {
    int r, c;
    if (!getIndex(x, y, &r, &c)) throw std::out_of_range("getUpdatedAtPosition: position outside the map");
    return updated.at(static_cast<size_t>(r) + static_cast<size_t>(c) * rows) > std::numeric_limits<float>::epsilon();
  }
};

inline artp_params toArtp(const Params& p) {
  artp_params a{};
  a.torso_length = p.robot.torso.length; a.torso_width = p.robot.torso.width; a.torso_height = p.robot.torso.height;
  a.torso_off_x = p.robot.torso.offset.x; a.torso_off_y = p.robot.torso.offset.y; a.torso_off_z = p.robot.torso.offset.z;
  a.feet_off_x = p.robot.feet.offset.x; a.feet_off_y = p.robot.feet.offset.y; a.feet_off_z = p.robot.feet.offset.z;
  a.reach_x = p.robot.feet.reach.x; a.reach_y = p.robot.feet.reach.y; a.reach_z = p.robot.feet.reach.z;
  a.unknown_space_untraversable = p.planner.unknown_space_untraversable ? 1 : 0;
  a.use_directional_cost = p.objectives.custom_path_length.use_directional_cost ? 1 : 0;
  a.max_lon_vel = p.objectives.custom_path_length.max_lon_vel;
  a.max_lat_vel = p.objectives.custom_path_length.max_lat_vel;
  a.max_ang_vel = p.objectives.custom_path_length.max_ang_vel;
  a.cost_w_energy = p.planner.prm_motion_cost.cost_weights.energy;
  a.cost_w_time = p.planner.prm_motion_cost.cost_weights.time;
  a.cost_w_risk = p.planner.prm_motion_cost.cost_weights.risk;
  a.risk_threshold = p.planner.prm_motion_cost.risk_threshold;
  a.device = p.device;
  return a;
}

// Owns the artp_handle; shared by the plugin objects below (the reference shares its checker the same way,
// path_length_objective.cpp:20: checker_(si->getStateValidityChecker())).
class Handle {
 public:
  explicit Handle(const ParamsConstPtr& params) : params_(params) {
    const artp_params a = toArtp(*params);
    if (artp_create(&a, &h_) != ARTP_OK) throw std::runtime_error(std::string("artp_create: ") + artp_last_error(nullptr));
  }
  ~Handle() { artp_destroy(h_); }
  Handle(const Handle&) = delete;
  Handle& operator=(const Handle&) = delete;
  artp_handle* get() const { return h_; }
  const Params& params() const { return *params_; }
  void check(int rc, const char* what) const {
    if (rc != ARTP_OK) throw std::runtime_error(std::string(what) + ": " + artp_last_error(h_));
  }
 private:
  ParamsConstPtr params_;
  artp_handle* h_{nullptr};
};
using HandlePtr = std::shared_ptr<Handle>;

// art_planner::StateValidityChecker (validity_checker.cpp:9-45).
class StateValidityChecker {
 public:
  explicit StateValidityChecker(const ParamsConstPtr& params) : handle_(std::make_shared<Handle>(params)) {}
  explicit StateValidityChecker(const HandlePtr& handle) : handle_(handle) {}

  void setMap(const std::shared_ptr<Map>& map) { map_ = map; }                 // validity_checker.cpp:20-23

  void updateHeightField() {                                                    // validity_checker.cpp:27-31
    if (!map_) throw std::runtime_error("updateHeightField: no map");
    handle_->check(artp_set_map(handle_->get(), map_->elevation.data(), map_->elevation_masked.data(), map_->rows, map_->cols,
                                map_->resolution, map_->position_x, map_->position_y), "artp_set_map");
  }

  bool hasMap() const { return artp_has_map(handle_->get()) != 0; }             // validity_checker.cpp:33-35

  // art_planner::estimateNormals (utils.cpp:213-324) as processors::Basic calls it (basic.cpp:47), on the device; fills
  // the map's normal_x/y/z and plane_fit_std_dev layers and keeps them resident for SE3FromSE2Sampler.
  void estimateNormals() {
    if (!map_) throw std::runtime_error("estimateNormals: no map");
    const Params& p = handle_->params();
    const size_t ncell = static_cast<size_t>(map_->rows) * map_->cols;
    map_->normal_x.resize(ncell); map_->normal_y.resize(ncell); map_->normal_z.resize(ncell);
    map_->plane_fit_std_dev.resize(ncell);
    handle_->check(artp_estimate_normals(handle_->get(), (p.robot.torso.length + p.robot.torso.width) * 0.25,
                                         map_->normal_x.data(), map_->normal_y.data(), map_->normal_z.data(),
                                         map_->plane_fit_std_dev.data()), "artp_estimate_normals");
  }

  bool isValid(const State* state) const {                                      // validity_checker.cpp:39-45
    uint8_t v = 0;
    handle_->check(artp_check_poses(handle_->get(), &state->x, 1, &v), "artp_check_poses");
    return v != 0;
  }

  // Batch form for the rejection-sampling loops (prm_motion_cost.cpp:171-194, lazy_prm_star_min_update.cpp:549-556).
  // Pose3FromSE3 casts every field to float first (utils.h:25-38); doing that cast here halves the PCIe traffic and
  // gives identical flags.
  void isValidBatch(const std::vector<State>& states, std::vector<uint8_t>* valid) const {
    std::vector<float> buf(7 * states.size());
    for (size_t i = 0; i < states.size(); ++i) {
      const double* s = &states[i].x;
      for (int k = 0; k < 7; ++k) buf[7 * i + k] = static_cast<float>(s[k]);
    }
    valid->resize(states.size());
    handle_->check(artp_check_poses_f32(handle_->get(), buf.data(), states.size(), valid->data()), "artp_check_poses_f32");
  }

  // computeCumulativeProbabilityDistribution (probability_distribution.cpp:20-46) on the device: fills the map's cum_prob /
  // cum_prob_rowwise layers from `sample_probability` (rows x cols, column-major) and keeps them resident for the sampler.
  void computeSampleCdf(const std::vector<float>& sample_probability) {
    if (!map_) throw std::runtime_error("computeSampleCdf: no map");
    const size_t ncell = static_cast<size_t>(map_->rows) * map_->cols;
    if (sample_probability.size() != ncell) throw std::invalid_argument("computeSampleCdf: layer size mismatch");
    map_->cum_prob.resize(ncell);
    map_->cum_prob_rowwise.resize(map_->rows);
    handle_->check(artp_compute_sample_cdf(handle_->get(), sample_probability.data(), map_->cum_prob.data(),
                                           map_->cum_prob_rowwise.data()), "artp_compute_sample_cdf");
  }

  // The rejection-sampling loop `do { sampleUniform(s) } while (!isValid(s))` (prm_motion_cost.cpp:171-194,
  // lazy_prm_star_min_update.cpp:549-556) in batches: draw `batch` candidates with the caller's sampler, check them in
  // one call, keep the valid ones in draw order; repeat until n_wanted states are collected or max_draws candidates
  // were drawn (the reference bounds the same loop by time). Returns the number of candidates drawn.
  template <class Sampler>   // void sampler(State* out)
  size_t sampleValidBatch(Sampler&& sampler, size_t n_wanted, size_t batch, size_t max_draws, std::vector<State>* out) const {
    out->clear();
    size_t drawn = 0;
    std::vector<State> cand;
    std::vector<uint8_t> valid;
    while (out->size() < n_wanted && drawn < max_draws) {
      const size_t m = std::min(batch, max_draws - drawn);
      cand.resize(m);
      for (size_t i = 0; i < m; ++i) sampler(&cand[i]);
      drawn += m;
      isValidBatch(cand, &valid);
      for (size_t i = 0; i < m && out->size() < n_wanted; ++i)
        if (valid[i]) out->push_back(cand[i]);
    }
    return drawn;
  }

  const HandlePtr& handle() const { return handle_; }

 private:
  HandlePtr handle_;
  std::shared_ptr<Map> map_;
};
using StateValidityCheckerPtr = std::shared_ptr<StateValidityChecker>;

// art_planner::SE3FromSE2Sampler (sampler.cpp:13-131): sampleUniform on the device, one candidate per Philox counter,
// and the rejection loop around it (prm_motion_cost.cpp:171-194) as one fused sample -> isValid -> compact call.
class SE3FromSE2Sampler {
 public:
  // bounds: SE3 position bounds x,y (planner.cpp:148-160); only read when !sample_from_distribution.
  SE3FromSE2Sampler(const StateValidityCheckerPtr& checker, const std::shared_ptr<Map>& map, uint64_t seed,
                    const double low[2], const double high[2])
      : checker_(checker), seed_(seed) {
    const auto& h = checker_->handle();
    const Params& p = h->params();
    artp_sampler_params sp{};
    sp.max_roll_pert = p.sampler.max_roll_pert; sp.max_pitch_pert = p.sampler.max_pitch_pert;
    sp.sample_from_distribution = p.sampler.sample_from_distribution ? 1 : 0;
    sp.low[0] = low[0]; sp.low[1] = low[1]; sp.high[0] = high[0]; sp.high[1] = high[1];
    h->check(artp_set_sampler(h->get(), &sp, map->normal_x.data(), map->normal_y.data(), map->normal_z.data(),
                              map->plane_fit_std_dev.data(), map->cum_prob.empty() ? nullptr : map->cum_prob.data(),
                              map->cum_prob_rowwise.empty() ? nullptr : map->cum_prob_rowwise.data()), "artp_set_sampler");
  }
  void sampleUniform(State* state) {                                             // sampler.cpp:82-131
    const auto& h = checker_->handle();
    do {   // uniform mode: a draw outside the map is a NaN candidate; samplePositionInMap (sampler.cpp:46-50) draws again
      h->check(artp_sample_states(h->get(), nullptr, seed_, next_, 1, &state->x, nullptr), "artp_sample_states");
      ++next_;
    } while (state->x != state->x);
  }
  // n states, none NaN: rejected (outside-map, uniform mode only) candidates are redrawn from the following counters of
  // the stream, like the reference's draw-again loop; the output keeps draw order.
  void sampleUniformBatch(size_t n, std::vector<State>* states) {
    states->clear();
    states->reserve(n);
    const auto& h = checker_->handle();
    std::vector<State> buf;
    while (states->size() < n) {
      const size_t m = n - states->size();
      buf.resize(m);
      h->check(artp_sample_states(h->get(), nullptr, seed_, next_, m, &buf[0].x, nullptr), "artp_sample_states");
      next_ += m;
      for (const State& s : buf) if (s.x == s.x) states->push_back(s);
    }
  }
  // Draws n_draw candidates, returns the valid ones in draw order (what n_draw iterations of
  // `do sampleUniform(s) while (!isValid(s))` would have accepted).
  void sampleValidBatch(size_t n_draw, std::vector<State>* valid) {
    valid->resize(n_draw);
    size_t n_valid = 0;
    const auto& h = checker_->handle();
    if (n_draw)
      h->check(artp_sample_valid(h->get(), seed_, next_, n_draw, &(*valid)[0].x, n_draw, &n_valid), "artp_sample_valid");
    next_ += n_draw;
    valid->resize(n_valid);
  }
  uint64_t nextIndex() const { return next_; }
 private:
  StateValidityCheckerPtr checker_;
  uint64_t seed_;
  uint64_t next_{0};
};

// ompl::base::MotionValidator as the reference uses it: discrete validation over isValid with nd segments.
class MotionValidator {
 public:
  MotionValidator(const StateValidityCheckerPtr& checker, int n_segments) : checker_(checker), nd_(n_segments) {}
  // valid(s2) && valid(interpolate(s1, s2, j/nd)) for j = 1..nd-1 (OMPL DiscreteMotionValidator::checkMotion)
  bool checkMotion(const State* s1, const State* s2) const {
    uint8_t v = 0;
    const auto& h = checker_->handle();
    h->check(artp_check_motions(h->get(), &s1->x, &s2->x, 1, nd_ - 1, &v), "artp_check_motions");
    return v != 0;
  }
  void checkMotionBatch(const std::vector<State>& s1, const std::vector<State>& s2, std::vector<uint8_t>* valid) const {
    if (s1.size() != s2.size()) throw std::invalid_argument("checkMotionBatch: size mismatch");
    valid->resize(s1.size());
    if (s1.empty()) return;
    const auto& h = checker_->handle();
    h->check(artp_check_motions(h->get(), &s1[0].x, &s2[0].x, s1.size(), nd_ - 1, valid->data()), "artp_check_motions");
  }
  // DiscreteMotionValidator::checkMotion(s1, s2, lastValid) with this validator's segment count: returns validity and,
  // for an invalid motion, lastValid.second = the parameter of the last valid state before the first invalid one in
  // OMPL's order (j = 1 .. nd-1, then s2); *last_valid (nullable) receives interpolate(s1, s2, that parameter).
  bool checkMotion(const State* s1, const State* s2, double* last_valid_t, State* last_valid) const {
    uint8_t v = 0;
    double t = 1.0;
    const int32_t nd = nd_;
    const auto& h = checker_->handle();
    h->check(artp_check_motions_segments(h->get(), &s1->x, &s2->x, 1, &nd, nullptr, &v, &t), "artp_check_motions_segments");
    if (!v) {
      if (last_valid_t) *last_valid_t = t;
      if (last_valid) *last_valid = interpolateSE3(*s1, *s2, t);
    }
    return v != 0;
  }
  // The batch form with PER-EDGE segment counts nd[e] = SE3StateSpace::validSegmentCount(s1, s2) (OMPL 1.4.2 rule,
  // artp_valid_segment_count) -- what si_->checkMotion does at prm_motion_cost.cpp:652 / lazy_prm_star_min_update.cpp:725.
  void checkMotionSegments(const std::vector<State>& s1, const std::vector<State>& s2, const artp_se3_space& space,
                           std::vector<uint8_t>* valid, std::vector<double>* last_valid_t, std::vector<int32_t>* nd = nullptr) const {
    if (s1.size() != s2.size()) throw std::invalid_argument("checkMotionSegments: size mismatch");
    valid->resize(s1.size());
    last_valid_t->resize(s1.size());
    if (s1.empty()) return;
    std::vector<int32_t> seg(s1.size());
    const auto& h = checker_->handle();
    h->check(artp_valid_segment_count(&space, &s1[0].x, &s2[0].x, s1.size(), seg.data()), "artp_valid_segment_count");
    h->check(artp_check_motions_segments(h->get(), &s1[0].x, &s2[0].x, s1.size(), seg.data(), nullptr, valid->data(),
                                         last_valid_t->data()), "artp_check_motions_segments");
    if (nd) *nd = seg;
  }
  // OMPL 1.4.2 SE3StateSpace::interpolate = RealVector lerp + SO3 slerp
  static State interpolateSE3(const State& a, const State& b, double t) {
    State o;
    o.x = a.x + (b.x - a.x) * t; o.y = a.y + (b.y - a.y) * t; o.z = a.z + (b.z - a.z) * t;
    const double dq = a.qx * b.qx + a.qy * b.qy + a.qz * b.qz + a.qw * b.qw;
    const double dqa = std::fabs(dq);
    const double theta = (dqa > 1.0 - 1e-9) ? 0.0 : std::acos(dqa);
    if (theta > std::numeric_limits<double>::epsilon()) {
      const double d = 1.0 / std::sin(theta), s0 = std::sin((1.0 - t) * theta);
      double s1 = std::sin(t * theta);
      if (dq < 0) s1 = -s1;
      o.qx = (a.qx * s0 + b.qx * s1) * d; o.qy = (a.qy * s0 + b.qy * s1) * d;
      o.qz = (a.qz * s0 + b.qz * s1) * d; o.qw = (a.qw * s0 + b.qw * s1) * d;
    } else {
      o.qx = a.qx; o.qy = a.qy; o.qz = a.qz; o.qw = a.qw;
    }
    return o;
  }
  // PRMMotionCost::addValidMilestone's connection loop (prm_motion_cost.cpp:341-372) for a batch of candidate edges:
  // n_interp[e] = (unsigned)(lateralDistance / max_lateral) interior states, valid_prefix[e] = how many leading ones are
  // valid; the connection holds iff valid_prefix[e] == n_interp[e].
  void checkEdgeInteriors(const std::vector<State>& s1, const std::vector<State>& s2, double max_lateral,
                          std::vector<int32_t>* n_interp, std::vector<int32_t>* valid_prefix) const {
    if (s1.size() != s2.size()) throw std::invalid_argument("checkEdgeInteriors: size mismatch");
    n_interp->resize(s1.size());
    valid_prefix->resize(s1.size());
    if (s1.empty()) return;
    for (size_t e = 0; e < s1.size(); ++e) {
      const double dx = s2[e].x - s1[e].x, dy = s2[e].y - s1[e].y;             // lateralDistance, utils.h:52-61
      (*n_interp)[e] = static_cast<int32_t>(static_cast<unsigned int>(std::sqrt(dx * dx + dy * dy) / max_lateral));
    }
    const auto& h = checker_->handle();
    h->check(artp_check_edge_interiors(h->get(), &s1[0].x, &s2[0].x, s1.size(), n_interp->data(), max_lateral,
                                       valid_prefix->data()), "artp_check_edge_interiors");
  }
 private:
  StateValidityCheckerPtr checker_;
  int nd_;
};

// art_planner::PathLengthObjective (path_length_objective.cpp:26-70).
class PathLengthObjective {
 public:
  explicit PathLengthObjective(const StateValidityCheckerPtr& checker) : checker_(checker) {}
  double motionCost(const State* s1, const State* s2) const {
    double c = 0;
    const auto& h = checker_->handle();
    h->check(artp_path_length_cost(h->get(), &s1->x, &s2->x, 1, &c), "artp_path_length_cost");
    return c;
  }
  double motionCostHeuristic(const State* s1, const State* s2) const {           // path_length_objective.cpp:58-70
    const double dx = s2->x - s1->x, dy = s2->y - s1->y, dz = s2->z - s1->z;
    return std::sqrt(dx * dx + dy * dy + dz * dz) / checker_->handle()->params().objectives.custom_path_length.max_lon_vel;
  }
  void motionCostBatch(const std::vector<State>& s1, const std::vector<State>& s2, std::vector<double>* cost) const {
    cost->resize(s1.size());
    if (s1.empty()) return;
    const auto& h = checker_->handle();
    h->check(artp_path_length_cost(h->get(), &s1[0].x, &s2[0].x, s1.size(), cost->data()), "artp_path_length_cost");
  }
 private:
  StateValidityCheckerPtr checker_;
};

// Row-major dynamic float matrix, the shape of MotionCostObjective::EdgeMatrix (motion_cost_objective.h:22).
struct EdgeMatrix {
  size_t n_rows{0}, n_cols{0};
  std::vector<float> v;
  void resize(size_t r, size_t c) { n_rows = r; n_cols = c; v.assign(r * c, 0.0f); }
  size_t rows() const { return n_rows; }
  float& operator()(size_t r, size_t c) { return v[r * n_cols + c]; }
  float operator()(size_t r, size_t c) const { return v[r * n_cols + c]; }
  const float* data() const { return v.data(); }
  float* data() { return v.data(); }
};

// art_planner::MotionCostObjective (motion_cost_objective.h:19-78, motion_cost_objective.cpp:28-95). The batch functor
// defaults to the in-process network (artp_motion_cost) instead of the ROS cost-server call of planner_ros.cpp:283-308.
class MotionCostObjective {
 public:
  using MotionCostFunc = std::function<bool(const EdgeMatrix&, EdgeMatrix*)>;

  explicit MotionCostObjective(const StateValidityCheckerPtr& checker, std::unique_ptr<MotionCostFunc> func = nullptr)
      : checker_(checker), motion_cost_func_(std::move(func)) {
    if (!motion_cost_func_) {
      HandlePtr h = checker_->handle();
      motion_cost_func_.reset(new MotionCostFunc([h](const EdgeMatrix& edges, EdgeMatrix* costs) {
        costs->resize(edges.rows(), 3);
        return artp_motion_cost(h->get(), edges.data(), edges.rows(), costs->data()) == ARTP_OK;
      }));
    }
  }
  void setWeights(const std::vector<float>& blob) {
    checker_->handle()->check(artp_set_cost_weights(checker_->handle()->get(), blob.data(), blob.size()), "artp_set_cost_weights");
  }
  void updateFeatures() { checker_->handle()->check(artp_update_features(checker_->handle()->get()), "artp_update_features"); }

  double getCost(const float* e3) const {                                        // motion_cost_objective.h:54-61
    const auto& w = checker_->handle()->params().planner.prm_motion_cost.cost_weights;
    // getEnergy/getTime/getRisk return double: the weighted sum is evaluated in double on exact float products
    return static_cast<double>(e3[0]) * w.energy + static_cast<double>(e3[1]) * w.time + static_cast<double>(e3[2]) * w.risk;
  }
  bool isFeasible(const float* e3) const {                                       // motion_cost_objective.h:63-65
    return static_cast<double>(e3[2]) <= checker_->handle()->params().planner.prm_motion_cost.risk_threshold;
  }
  bool costQuery(const EdgeMatrix& edge_matrix, EdgeMatrix* edge_cost) const {   // motion_cost_objective.cpp:28-33
    edge_cost->resize(edge_matrix.rows(), 3);
    return (*motion_cost_func_)(edge_matrix, edge_cost);
  }

  // motion_cost_objective.cpp:36-95: split the edge at max_query_edge_length, query every piece, sum; +inf if any piece
  // is too risky; throws "Motion cost call failed" if the functor fails.
  double motionCost(const State* s1, const State* s2) const {
    const double dx = s2->x - s1->x, dy = s2->y - s1->y;
    const double dist = std::sqrt(dx * dx + dy * dy);                            // lateralDistance, utils.h:52-61
    const auto& pm = checker_->handle()->params().planner.prm_motion_cost;
    const unsigned n_interp = static_cast<unsigned>(dist / pm.max_query_edge_length);
    const double n_interp_div = 1.0 / (n_interp + 1);
    EdgeMatrix em, ec;
    em.resize(n_interp + 1, 6);
    em(0, 3) = static_cast<float>(s1->x); em(0, 4) = static_cast<float>(s1->y); em(0, 5) = yaw(*s1);
    em(n_interp, 0) = static_cast<float>(s2->x); em(n_interp, 1) = static_cast<float>(s2->y); em(n_interp, 2) = yaw(*s2);
    for (unsigned step = 1; step < n_interp + 1; ++step) {
      const State cur = interpolate(*s1, *s2, step * n_interp_div);
      em(step - 1, 0) = static_cast<float>(cur.x); em(step - 1, 1) = static_cast<float>(cur.y); em(step - 1, 2) = yaw(cur);
      em(step, 3) = static_cast<float>(cur.x); em(step, 4) = static_cast<float>(cur.y); em(step, 5) = yaw(cur);
    }
    if (!costQuery(em, &ec)) throw std::runtime_error("Motion cost call failed");
    double cost = 0;
    for (unsigned i = 0; i < n_interp + 1; ++i) {
      const float* e3 = ec.data() + 3 * i;
      if (static_cast<double>(e3[2]) > pm.risk_threshold) return std::numeric_limits<double>::infinity();
      cost += getCost(e3);
    }
    return cost;
  }
  double motionCostHeuristic(const State*, const State*) const { return 0.0; }   // motion_cost_objective.cpp:99-103

  // PRMMotionCostMaintainer::updateEdges / computeCostForVertexEdges (prm_motion_cost.cpp:27-128) for a batch of graph
  // edges (source = v1, target = v2): edge matrix -> cost query -> per edge isFeasible ? getCost : +inf, in one device call.
  // Returns false where the reference's functor would (then the graph is left alone, :69-72 / :124-127).
  bool updateEdgesBatch(const std::vector<State>& source, const std::vector<State>& target, std::vector<double>* cost,
                        std::vector<uint8_t>* feasible) const {
    if (source.size() != target.size()) throw std::invalid_argument("updateEdgesBatch: size mismatch");
    cost->resize(source.size());
    feasible->resize(source.size());
    if (source.empty()) return true;
    return artp_motion_cost_states(checker_->handle()->get(), &source[0].x, &target[0].x, source.size(), cost->data(),
                                   feasible->data(), nullptr) == ARTP_OK;
  }

  // getYawFromSO3 (utils.h:80-88): double atan2 returned through float
  static float yaw(const State& s) {
    return static_cast<float>(std::atan2(2 * (s.qw * s.qz + s.qx * s.qy), 1 - 2 * (s.qy * s.qy + s.qz * s.qz)));
  }
  // OMPL 1.4.2 SE3StateSpace::interpolate = RealVector lerp + SO3 slerp
  static State interpolate(const State& a, const State& b, double t) {
    State o;
    o.x = a.x + (b.x - a.x) * t; o.y = a.y + (b.y - a.y) * t; o.z = a.z + (b.z - a.z) * t;
    const double dq = a.qx * b.qx + a.qy * b.qy + a.qz * b.qz + a.qw * b.qw;
    const double dqa = std::fabs(dq);
    const double theta = (dqa > 1.0 - 1e-9) ? 0.0 : std::acos(dqa);
    if (theta > std::numeric_limits<double>::epsilon()) {
      const double d = 1.0 / std::sin(theta), s0 = std::sin((1.0 - t) * theta);
      double s1 = std::sin(t * theta);
      if (dq < 0) s1 = -s1;
      o.qx = (a.qx * s0 + b.qx * s1) * d; o.qy = (a.qy * s0 + b.qy * s1) * d;
      o.qz = (a.qz * s0 + b.qz * s1) * d; o.qw = (a.qw * s0 + b.qw * s1) * d;
    } else {
      o.qx = a.qx; o.qy = a.qy; o.qz = a.qz; o.qw = a.qw;
    }
    return o;
  }

 private:
  StateValidityCheckerPtr checker_;
  std::unique_ptr<MotionCostFunc> motion_cost_func_;
};

namespace processors {
// processors::computeChange (change.cpp:9-51) on the device: fills map_new->updated (1 where the height changed by more
// than height_change_for_update or the traversability went 1 -> 0 over the overlap of the two maps, and everywhere
// outside it). The layer also stays on the handle, bit-packed, for LazyPRMStarMinUpdateMaintainer.
inline void computeChange(const HandlePtr& handle, const std::shared_ptr<Map>& map_new, const std::shared_ptr<Map>& map_old,
                          float height_change_for_update) {
  auto grid = [](const Map& m, const char* which) {
    const size_t ncell = static_cast<size_t>(m.rows) * m.cols;
    if (m.elevation.size() != ncell || m.traversability_thresholded.size() != ncell)
      throw std::invalid_argument(std::string("computeChange: ") + which + " map needs elevation and traversability_thresholded");
    artp_grid g{};
    g.elevation = m.elevation.data(); g.traversability_thresholded = m.traversability_thresholded.data();
    g.rows = m.rows; g.cols = m.cols; g.res = m.resolution; g.cx = m.position_x; g.cy = m.position_y;
    return g;
  };
  const artp_grid gn = grid(*map_new, "new"), go = grid(*map_old, "old");
  map_new->updated.resize(static_cast<size_t>(map_new->rows) * map_new->cols);
  handle->check(artp_compute_change(handle->get(), &gn, &go, height_change_for_update, map_new->updated.data()),
                "artp_compute_change");
}
}  // namespace processors

// LazyPRMStarMinUpdateMaintainer::update (lazy_prm_star_min_update.cpp:123-135) for a roadmap given as arrays, against
// the change layer of the last processors::computeChange on the same handle. The per-vertex / per-edge questions run in
// one device call; the Boost graph surgery (removeVertices, components, start / goal re-insertion) stays with the planner.
class LazyPRMStarMinUpdateMaintainer {
 public:
  static constexpr unsigned int VALIDITY_UNKNOWN = 0, VALIDITY_TRUE = 1;   // ompl::geometric::LazyPRM's flags
  explicit LazyPRMStarMinUpdateMaintainer(const HandlePtr& handle) : handle_(handle) {}

  // edges: 2 vertex indices per edge (boost::source, boost::target). Returns the vertices removeOutdatedVertices
  // (:58-72) removes -- those outside the new map -- in ascending order; their edges go with them. Then, when
  // invalidate_updated_graph_components is set, invalidateUpdatedGraphComponents (:18-54) on what stays: every
  // VALIDITY_TRUE vertex on an updated cell and every VALIDITY_TRUE edge whose grid line crosses one becomes
  // VALIDITY_UNKNOWN. Other flags are left as they are.
  std::vector<size_t> update(const std::vector<State>& vertices, std::vector<unsigned int>* vertex_validity,
                             const std::vector<uint32_t>& edges, std::vector<unsigned int>* edge_validity,
                             bool invalidate_updated_graph_components = true) const {
    const size_t nv = vertices.size(), ne = edges.size() / 2;
    if (edges.size() % 2 || vertex_validity->size() != nv || edge_validity->size() != ne)
      throw std::invalid_argument("LazyPRMStarMinUpdateMaintainer::update: size mismatch");
    std::vector<uint8_t> vf(nv), ef(ne);
    handle_->check(artp_roadmap_updates(handle_->get(), nv ? &vertices[0].x : nullptr, nv, ne ? edges.data() : nullptr, ne,
                                        vf.data(), ef.data()), "artp_roadmap_updates");
    std::vector<size_t> removed;
    for (size_t v = 0; v < nv; ++v) {
      if (vf[v] == 2) { removed.push_back(v); continue; }
      unsigned int& vd = (*vertex_validity)[v];
      if (invalidate_updated_graph_components && (vd & VALIDITY_TRUE) && vf[v] == 1) vd = VALIDITY_UNKNOWN;
    }
    if (invalidate_updated_graph_components)
      for (size_t e = 0; e < ne; ++e) {
        unsigned int& ed = (*edge_validity)[e];
        if ((ed & VALIDITY_TRUE) && ef[e] == 1) ed = VALIDITY_UNKNOWN;
      }
    return removed;
  }

 private:
  HandlePtr handle_;
};

}  // namespace artp_host

#ifdef ARTP_WITH_OMPL
// OMPL adapters (compiled only where OMPL >= 1.4.2 is installed): the exact plugin surface of planner.cpp:125-130.
#include <ompl/base/MotionValidator.h>
#include <ompl/base/SpaceInformation.h>
#include <ompl/base/StateValidityChecker.h>
#include <ompl/base/objectives/PathLengthOptimizationObjective.h>
#include <ompl/base/spaces/SE3StateSpace.h>
namespace artp_host {
namespace ob = ompl::base;
inline State fromOmpl(const ob::State* s) {
  const auto* se3 = s->as<ob::SE3StateSpace::StateType>();
  State o;
  o.x = se3->getX(); o.y = se3->getY(); o.z = se3->getZ();
  o.qx = se3->rotation().x; o.qy = se3->rotation().y; o.qz = se3->rotation().z; o.qw = se3->rotation().w;
  return o;
}
class OmplStateValidityChecker : public ob::StateValidityChecker {
 public:
  OmplStateValidityChecker(const ob::SpaceInformationPtr& si, const StateValidityCheckerPtr& c) : ob::StateValidityChecker(si), c_(c) {}
  bool isValid(const ob::State* state) const override { const State s = fromOmpl(state); return c_->isValid(&s); }
 private:
  StateValidityCheckerPtr c_;
};
class OmplMotionValidator : public ob::MotionValidator {
 public:
  OmplMotionValidator(const ob::SpaceInformationPtr& si, const StateValidityCheckerPtr& c) : ob::MotionValidator(si), c_(c) {}
  bool checkMotion(const ob::State* s1, const ob::State* s2) const override {
    const State a = fromOmpl(s1), b = fromOmpl(s2);
    return MotionValidator(c_, si_->getStateSpace()->validSegmentCount(s1, s2)).checkMotion(&a, &b);
  }
  bool checkMotion(const ob::State* s1, const ob::State* s2, std::pair<ob::State*, double>& lastValid) const override {
    const State a = fromOmpl(s1), b = fromOmpl(s2);
    double t = 1.0;
    const bool ok = MotionValidator(c_, si_->getStateSpace()->validSegmentCount(s1, s2)).checkMotion(&a, &b, &t, nullptr);
    if (!ok) {   // DiscreteMotionValidator: lastValid is only written for invalid motions
      lastValid.second = t;
      if (lastValid.first) si_->getStateSpace()->interpolate(s1, s2, t, lastValid.first);
    }
    return ok;
  }
 private:
  StateValidityCheckerPtr c_;
};
class OmplPathLengthObjective : public ob::PathLengthOptimizationObjective {
 public:
  OmplPathLengthObjective(const ob::SpaceInformationPtr& si, const StateValidityCheckerPtr& c)
      : ob::PathLengthOptimizationObjective(si), o_(c) {}
  ob::Cost motionCost(const ob::State* s1, const ob::State* s2) const override {
    const State a = fromOmpl(s1), b = fromOmpl(s2);
    return ob::Cost(o_.motionCost(&a, &b));
  }
 private:
  PathLengthObjective o_;
};
}  // namespace artp_host
#endif
