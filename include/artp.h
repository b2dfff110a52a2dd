/*
 * include/artp.h -- C ABI of the B200-native art_planner hot path (libartp.so).
 *
 * Drop-in boundary (SURVEY.md section 8b): everything the reference's OMPL plugins for this path need,
 * as plain C: pointers + sizes, no C++/torch types, no exceptions across the boundary. Every entry point
 * returns 0 on success or a negative ARTP_E_* code; artp_last_error() gives the message.
 * There is NO CPU fallback: if no CUDA device / kernel image is usable the calls fail with ARTP_E_CUDA.
 *
 * Reference interfaces each entry point replaces (paths relative to the reference tree):
 *   artp_create / artp_destroy      art_planner::StateValidityChecker ctor (validity_checker.cpp:9-16) ->
 *                                   ValidityCheckerBody/Feet ctors -> HeightMapBoxChecker ctor
 *                                   (height_map_box_checker.cpp:11-26); parameters from art_planner::Params
 *                                   (include/art_planner/params.h:14-123)
 *   artp_set_map                    StateValidityChecker::setMap + updateHeightField (validity_checker.cpp:20-31)
 *                                   -> HeightMapBoxChecker::setHeightField (height_map_box_checker.cpp:38-54);
 *                                   installed at Planner::setMap (art_planner/src/planner.cpp:135-163)
 *   artp_check_poses[_device]       ompl::base::StateValidityChecker::isValid, i.e.
 *                                   art_planner::StateValidityChecker::isValid (validity_checker.cpp:39-45)
 *   artp_check_motions[_device]     ompl::base::MotionValidator::checkMotion as the reference uses it: OMPL's
 *                                   DiscreteMotionValidator over isValid (call sites prm_motion_cost.cpp:652,
 *                                   lazy_prm_star_min_update.cpp:725) and the in-tree interpolation loop
 *                                   PRMMotionCost::addValidMilestone (prm_motion_cost.cpp:341-372)
 *   artp_check_edge_interiors[_device]  that same addValidMilestone loop with its exact semantics: per-edge
 *                                   interior-state counts, no endpoint check, stop at the first invalid state
 *   artp_set_sampler, artp_sample_states[_device], artp_sample_valid[_device], artp_sampler_uniforms
 *                                   ompl::base::StateSampler::sampleUniform -> SE3FromSE2Sampler::sampleUniform
 *                                   (src/sampler.cpp:82-131, positions :40-77) and the rejection loops around it
 *                                   (prm_motion_cost.cpp:171-194, lazy_prm_star_min_update.cpp:549-556)
 *   artp_estimate_normals           art_planner::estimateNormals (src/utils.cpp:213-324; processors::Basic, basic.cpp:47)
 *   artp_compute_sample_cdf         computeCumulativeProbabilityDistribution
 *                                   (src/map/processors/probability_distribution.cpp:20-46)
 *   artp_compact_valid_device, artp_pack_valid_bits_device, artp_compact_bits_device
 *                                   no reference counterpart: the multi-GPU verdict exchange (SURVEY 8e)
 *   artp_path_length_cost[_device]  ompl::base::OptimizationObjective::motionCost ->
 *                                   PathLengthObjective::motionCost (objectives/path_length_objective.cpp:26-70)
 *   artp_set_cost_weights, artp_update_features, artp_motion_cost[_device]
 *                                   the MotionCostFunc batch functor (objectives/motion_cost_objective.h:22-23)
 *                                   = ROS service cost_query (art_planner_ros/src/planner_ros.cpp:283-308,
 *                                   art_planner_motion_cost/scripts/cost_query_server.py:145-169,
 *                                   predictor/predictor.py:28-44, predictor/cost_query.py:39-69)
 *   artp_combine_cost               MotionCostObjective::getCost / isFeasible (motion_cost_objective.h:54-66)
 *   artp_compute_change[_device]    processors::computeChange (src/map/processors/change.cpp:9-51), the old-map processor
 *                                   Planner::setUpMapProcessors installs when invalidate_updated_graph_components is set
 *                                   (planner.cpp:60-69)
 *   artp_roadmap_updates[_device]   the per-vertex / per-edge questions of LazyPRMStarMinUpdateMaintainer::update
 *                                   (lazy_prm_star_min_update.cpp:123-135): isOutOfBounds for removeOutdatedVertices
 *                                   (:58-72, :94-98) and wasUpdated(v) / wasUpdated(e) for invalidateUpdatedGraphComponents
 *                                   (:18-54, :76-91) = Map::getUpdatedAtPosition / getUpdatedOnLine (map.h:86-89,
 *                                   map.cpp:44-53)
 */
#ifndef ARTP_H
#define ARTP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ARTP_OK            0
#define ARTP_E_INVALID    -1   /* bad argument */
#define ARTP_E_NOMAP      -2   /* no map set (hasMap() == false) */
#define ARTP_E_CUDA       -3   /* CUDA runtime error / no device */
#define ARTP_E_LIMIT      -4   /* box/map combination exceeds a compiled limit */
#define ARTP_E_NOWEIGHTS  -5   /* motion-cost network weights / features not set */
#define ARTP_E_WINDOW     -6   /* a box reached outside the handle's map window (artp_set_map_window) */

/* art_planner::Params fields the hot path reads (include/art_planner/params.h). Doubles as in the reference. */
typedef struct artp_params {
  double torso_length, torso_width, torso_height;   /* params.h:92-94   */
  double torso_off_x, torso_off_y, torso_off_z;     /* params.h:96-100  */
  double feet_off_x, feet_off_y, feet_off_z;        /* params.h:106-110 */
  double reach_x, reach_y, reach_z;                 /* params.h:112-116 */
  int    unknown_space_untraversable;               /* params.h:26      */
  int    use_directional_cost;                      /* params.h:73      */
  double max_lon_vel, max_lat_vel, max_ang_vel;     /* params.h:74-76   */
  float  cost_w_energy, cost_w_time, cost_w_risk;   /* params.h:57-61   */
  float  risk_threshold;                            /* params.h:55      */
  int    device;                                    /* CUDA device ordinal for this handle */
} artp_params;

typedef struct artp_handle artp_handle;

typedef struct artp_stats {
  uint64_t poses_checked;      /* pose checks executed since creation */
  uint64_t poses_deferred;     /* deferred items summed over the calls whose stats were read (one read per call) */
  uint64_t kernel_launches;    /* kernels launched by this handle since creation */
  uint32_t last_deferred;      /* deferred count of the most recent check call */
  uint32_t last_launches;      /* kernels launched by the most recent call */
  uint32_t last_queued_boxes;  /* boxes the classify stage queued for the later stages in the most recent call's last round */
  uint32_t last_queued_warp_stage;   /* ... of which in the big-tile queue (torso boxes, reach boxes of unusual size) */
  uint32_t last_queued_reach_stage;  /* ... of which in the one-warp-per-box reach queue (zones with -inf or mergeable planes) */
  uint32_t last_reach_plane_stage;   /* ... of which in the 8-lane-group reach queue (all-finite, merge-free zones) */
} artp_stats;

int  artp_create(const artp_params* params, artp_handle** out);
void artp_destroy(artp_handle* h);
const char* artp_last_error(const artp_handle* h);   /* h may be NULL: last creation error */

/* Layers are HOST pointers in grid_map layout: column-major rows x cols floats, (i,j) at data[i + j*rows];
 * lengths = rows*res, cols*res; centre (cx, cy). Heights must be finite or -inf. */
int artp_set_map(artp_handle* h, const float* elevation, const float* elevation_masked,
                 int rows, int cols, double res, double cx, double cy);
int artp_has_map(const artp_handle* h);
/* Spatial shard of a map (multi-GPU, SURVEY 8e): the handle receives only rows [row0, row0 + nrows) of the rows x cols
 * layers (HOST pointers to nrows x cols column-major matrices; row0 a multiple of 4) -- its slab plus a halo of at least
 * the largest box half-diagonal + box offsets -- while rows, res, cx, cy describe the FULL map. Geometry (ODE sample
 * spacing L / (N - 1), vertex coordinates, grid_map isInside) is that of the full map, so verdicts are bit-identical to a
 * handle holding everything; device memory and the range / plane tables shrink to the window. A pose whose boxes reach
 * outside the window is reported invalid and raises ARTP_E_WINDOW (sticky, like ARTP_E_LIMIT): route every sample to
 * the shard that holds it. The sampler, normal estimation and the cost network need the whole map (ARTP_E_INVALID). */
int artp_set_map_window(artp_handle* h, const float* elevation, const float* elevation_masked, int rows, int cols,
                        double res, double cx, double cy, int row0, int nrows);

/* n SE(3) states, 7 doubles each (x y z qx qy qz qw) -> valid[n] (0/1). HOST buffers; H2D/D2H inside. */
int artp_check_poses(artp_handle* h, const double* states, size_t n, uint8_t* valid);
/* Same with DEVICE buffers on `stream` (a cudaStream_t cast to void*, may be NULL); asynchronous. */
int artp_check_poses_device(artp_handle* h, const double* d_states, size_t n, uint8_t* d_valid, void* stream);

/* Pinned host memory for the adapter's batch buffers (states in, verdicts out): pages from cudaHostAlloc reach the device
 * at PCIe line rate, which memory pinned after the fact does not (profiles/pcie_probe.cu). NULL on failure. */
void* artp_host_alloc(size_t bytes);
void  artp_host_free(void* p);

/* float32 states (n x 7 floats): the caller applies the double -> float cast Pose3FromSE3 (utils.h:25-38) performs
 * first; results are identical to the double entry points at half the host<->device traffic. */
int artp_check_poses_f32(artp_handle* h, const float* states, size_t n, uint8_t* valid);
int artp_check_poses_f32_device(artp_handle* h, const float* d_states, size_t n, uint8_t* d_valid, void* stream);

/* Edge validity: valid(s2) && valid(interp(s1,s2,j/(n_steps+1))) for j = 1..n_steps (n_steps >= 0). */
int artp_check_motions(artp_handle* h, const double* s1, const double* s2, size_t n, int n_steps, uint8_t* valid);
int artp_check_motions_device(artp_handle* h, const double* d_s1, const double* d_s2, size_t n, int n_steps,
                              uint8_t* d_valid, void* stream);

/* ompl::base::DiscreteMotionValidator::checkMotion(s1, s2[, lastValid]) (OMPL 1.4.2; the reference's default motion
 * validator, call sites prm_motion_cost.cpp:652, lazy_prm_star_min_update.cpp:725) with PER-EDGE segment counts:
 * edge e is valid iff interpolate(s1, s2, j / nd[e]) is valid for j = 1 .. nd[e]-1 and s2 is valid. nd[e] =
 * SE3StateSpace::validSegmentCount(s1, s2); nd == NULL: computed by artp_valid_segment_count from *sp (the space
 * parameters Planner::setMap installs, planner.cpp:146-156). last_valid_t (nullable) receives lastValid.second: the
 * parameter of the last valid state before the first invalid one in OMPL's order ((j-1)/nd, or (nd-1)/nd when only s2
 * is invalid; 1.0 for valid edges) -- the caller obtains lastValid.first by interpolating at that parameter. */
typedef struct artp_se3_space {
  double low[3], high[3];                  /* RealVectorBounds of the SE3 space (planner.cpp:148-156) */
  double longest_valid_segment_fraction;   /* OMPL default 0.01 (the reference never changes it); <= 0 means 0.01 */
} artp_se3_space;
int artp_valid_segment_count(const artp_se3_space* sp, const double* s1, const double* s2, size_t n, int32_t* nd);
int artp_check_motions_segments(artp_handle* h, const double* s1, const double* s2, size_t n, const int32_t* nd,
                                const artp_se3_space* sp, uint8_t* valid, double* last_valid_t);

/* PRMMotionCost::addValidMilestone's connection test (prm_motion_cost.cpp:341-372), batched over the n candidate
 * edges of new milestones: edge e has n_interp[e] interior states at t = step * (1.0 / (n_interp[e] + 1)),
 * step = 1..n_interp[e] (endpoints are NOT checked there), and the reference loop stops at the first invalid one.
 * valid_prefix[e] = number of leading valid interior states; the connection is valid iff it equals n_interp[e], and
 * the caller inserts the first valid_prefix[e] states as intermediate milestones exactly like :356-366.
 * n_interp == NULL: computed per edge as (unsigned)(lateralDistance(s1, s2) / max_lateral) like :341-343
 * (the reference's max_lateral is 0.5). Total interior states must be < 2^32. */
int artp_check_edge_interiors(artp_handle* h, const double* s1, const double* s2, size_t n, const int32_t* n_interp,
                              double max_lateral, int32_t* valid_prefix);
/* DEVICE buffers: d_item_off = n + 1 exclusive prefix sums (uint32) of the per-edge interior-state counts,
 * total_items = d_item_off[n], d_item_valid = scratch of total_items bytes that receives the per-state flags. */
int artp_check_edge_interiors_device(artp_handle* h, const double* d_s1, const double* d_s2, size_t n,
                                     const uint32_t* d_item_off, size_t total_items, uint8_t* d_item_valid,
                                     int32_t* d_valid_prefix, void* stream);

/* ---- SE3FromSE2Sampler::sampleUniform (art_planner/src/sampler.cpp:40-131) on the device ------------------------
 * SURVEY 8(f) rank 2: candidates are generated where they are checked, so the rejection loops
 * (prm_motion_cost.cpp:171-194, lazy_prm_star_min_update.cpp:549-556) need no host->device pose stream.
 * One candidate consumes six uniform01 variates in the order the reference draws them:
 *   sample_from_distribution:  u0 = samp_col, u1 = samp_row (:56-57), u2 -> uniformReal(-1,1) (:103),
 *                              u3,u4,u5 -> RNG::eulerRPY roll, pitch, yaw (:114)
 *   otherwise:                 u0 -> x, u1 -> y in [low, high]; a position outside the map is a rejected candidate
 *                              (NaN state, rowcol -1, never valid) where the reference loop (:46-50) draws again.
 * The variates are either caller-provided (u != NULL) or produced by the documented counter-based stream
 * Philox4x32-10(key = seed, counter = (sample index, block 0..2, "ARTP")), see artp_sampler_uniforms(). */
typedef struct artp_sampler_params {
  double max_roll_pert, max_pitch_pert;   /* params.h:79-80, radians */
  int    sample_from_distribution;        /* params.h:81 */
  double low[2], high[2];                 /* SE3 position bounds x,y (planner.cpp:148-160); uniform mode only */
} artp_sampler_params;

/* Per-cell layers the sampler reads, HOST pointers in grid_map layout (like artp_set_map, which must come first and
 * provides "elevation" and the geometry): normal_x/y/z, plane_fit_std_dev (Map::getNormal / getPlaneFitStdDev,
 * map.h:94-116), "cum_prob" and column 0 of "cum_prob_rowwise_hack" (probability_distribution.cpp:20-46; may be NULL
 * when !sample_from_distribution). The four normal / plane-fit pointers may all be NULL after artp_estimate_normals.
 * CDF rows must be non-decreasing or all NaN (else ARTP_E_INVALID).
 * artp_set_map invalidates the sampler layers. */
/* art_planner::estimateNormals (art_planner/src/utils.cpp:213-324; called from processors::Basic, basic.cpp:47, with
 * estimation_radius = (torso.length + torso.width) * 0.25) for the elevation layer of the current map, on the device.
 * The four layers stay on the device as the sampler's normal / plane-fit layers (then artp_set_sampler may be called
 * with the four pointers NULL) and are copied to the non-NULL HOST outputs (grid_map layout). Bit-identical to the
 * reference's float arithmetic (the elevation layer's -0 is stored as +0, see artp_set_map). */
int artp_estimate_normals(artp_handle* h, double estimation_radius, float* normal_x, float* normal_y, float* normal_z,
                          float* plane_fit_std_dev);
/* computeCumulativeProbabilityDistribution (src/map/processors/probability_distribution.cpp:20-46) on the device:
 * "sample_probability" (HOST, grid_map layout) -> "cum_prob" and column 0 of "cum_prob_rowwise_hack", kept on the device
 * as the sampler's CDF layers (artp_set_sampler may then get NULL for both) and copied to the non-NULL HOST outputs.
 * Sums run left to right per row; rows without mass become NaN rows exactly like the reference's 0/0. */
int artp_compute_sample_cdf(artp_handle* h, const float* sample_probability, float* cum_prob, float* cum_prob_rowwise);
int artp_set_sampler(artp_handle* h, const artp_sampler_params* sp, const float* normal_x, const float* normal_y,
                     const float* normal_z, const float* plane_fit_std_dev, const float* cum_prob,
                     const float* cum_prob_rowwise);
/* The variates of samples first_sample .. first_sample+n-1 under `seed`: u[n][6] (host). */
int artp_sampler_uniforms(artp_handle* h, uint64_t seed, uint64_t first_sample, size_t n, double* u);
/* n candidates -> states[n][7] (x y z qx qy qz qw), rowcol[n][2] (sampled cell; nullable). u == NULL: Philox stream. */
int artp_sample_states(artp_handle* h, const double* u, uint64_t seed, uint64_t first_sample, size_t n, double* states,
                       int32_t* rowcol);
int artp_sample_states_device(artp_handle* h, const double* d_u, uint64_t seed, uint64_t first_sample, size_t n,
                              double* d_states, int32_t* d_rowcol, void* stream);
/* Fused sample -> isValid -> ordered compaction: draws candidates first_sample .. first_sample+n_draw-1 of the Philox
 * stream and writes the valid ones, in draw order, to states (at most `capacity`); *n_valid / *d_count = number of
 * valid candidates (> capacity: output truncated). */
int artp_sample_valid(artp_handle* h, uint64_t seed, uint64_t first_sample, size_t n_draw, double* states,
                      size_t capacity, size_t* n_valid);
int artp_sample_valid_device(artp_handle* h, uint64_t seed, uint64_t first_sample, size_t n_draw, double* d_states_out,
                             size_t capacity, uint32_t* d_count, void* stream);

/* PathLengthObjective::motionCost for n edges -> cost[n] (double). */
int artp_path_length_cost(artp_handle* h, const double* s1, const double* s2, size_t n, double* cost);
int artp_path_length_cost_device(artp_handle* h, const double* d_s1, const double* d_s2, size_t n,
                                 double* d_cost, void* stream);

/* Ordered compaction of a validity mask into indices (for the multi-GPU index all-gather):
 * d_indices[k] = base + i for the k-th i with d_valid[i] != 0; *d_count = number written. Device buffers. */
int artp_compact_valid_device(artp_handle* h, const uint8_t* d_valid, size_t n, int64_t base,
                              int64_t* d_indices, uint32_t* d_count, void* stream);
/* Multi-GPU exchange format: the mask bit-packed (item i = bit i&31 of word i>>5; (n+31)/32 words, tail bits 0) --
 * 125 KB per 10^6 poses on the wire instead of 8 MB of padded indices -- and the ordered compaction of such a
 * (gathered) bit mask, which every rank runs on the all-gathered words to obtain the global valid-index list. */
int artp_pack_valid_bits_device(artp_handle* h, const uint8_t* d_valid, size_t n, uint32_t* d_bits, void* stream);
/* A shard's step of the multi-GPU path in one call: isValid of its n samples (d_valid, bytes) and the bit-packed mask
 * (d_bits, (n+31)/32 words) that goes on the wire. */
int artp_check_poses_bits_device(artp_handle* h, const double* d_states, size_t n, uint8_t* d_valid, uint32_t* d_bits, void* stream);
/* Ordered compaction into 32-bit indices (base + i): the per-shard valid-sample list; a consumer that needs the global
 * list reads the per-rank counts + segments. */
int artp_compact_valid_u32_device(artp_handle* h, const uint8_t* d_valid, size_t n, uint32_t base, uint32_t* d_indices,
                                  uint32_t* d_count, void* stream);
int artp_compact_bits_device(artp_handle* h, const uint32_t* d_bits, size_t n, int64_t base, int64_t* d_indices,
                             uint32_t* d_count, void* stream);

int artp_get_stats(artp_handle* h, artp_stats* out);

/* Threads and streams. A handle is safe to share between threads (the reference's checkers are called from the planning
 * thread, the ROS callback threads and the cleaner thread, SURVEY 8b): every entry point holds the handle's lock for its
 * whole duration, host-buffer calls including their staging copies. The *_device entry points are asynchronous on the
 * caller's stream; calls issued on DIFFERENT streams are ordered against each other on the device (each waits for the
 * previous user of the handle's scratch buffers), so they are safe but do not overlap -- use one handle per stream for
 * concurrency.
 *
 * Errors detected on the device: if the plane-grouping stage cannot hold a zone in its shared-memory store (sized at
 * artp_set_map from the box diagonals; cannot happen for boxes that passed artp_set_map unless the test hook below is
 * used) the affected pose / edge is reported INVALID (fail closed) and a sticky error is raised: host-buffer calls return
 * ARTP_E_LIMIT from the call that caused it; after asynchronous *_device calls, synchronise the stream and call
 * artp_poll_error (returns ARTP_E_LIMIT once, then clears). artp_get_stats reports it too. artp_roadmap_updates_device
 * raises the same sticky error for an edge index >= nv; it is reported as ARTP_E_INVALID. */
int artp_poll_error(artp_handle* h);
/* Test hook: cap the plane store at max_triangles (0 = no cap) from the next artp_set_map on. */
int artp_debug_set_group_capacity(artp_handle* h, int max_triangles);

/* Environment switches (read at artp_create unless noted; experiments and A/B measurements, never needed in production):
 *   ARTP_NO_GROUPS=1        (read at artp_set_map) every undecided reach box takes the one-warp-per-box queue instead of the
 *                           8-lane-group kernel -- same verdicts (tests/test_pose_gpu.py runs both)
 *   ARTP_SLICE_ITEMS=n      host-buffer calls: equal H2D slices of n states instead of the built-in schedules
 *   ARTP_SLICE_SCHEDULE=a,b,...  host-buffer calls: slice fractions of a round (e.g. 0.1,0.2,0.3,0.4)
 *   ARTP_TRACE=1            host-buffer calls print the GPU timeline of their slices (copy landed, classify, box stages)
 *   ARTP_K0_FLAGS=2         classify stage without its reach-box vertex probes (measured slower: the boxes land in the queues)
 *   ARTP_FORK_ITEMS=n       rounds of up to n items run their three box kernels side by side on internal streams
 *                           (default: always; 0 = serial order)
 *   ARTP_PIPE_CAPS=g,f      host-buffer calls: grid caps of the per-slice reach kernels in half SM counts (default 4,4)
 * artp_set_timing(h, 1) makes the host-buffer calls run their slices back to back (the per-stage events need one stream):
 * leave it off when measuring end-to-end throughput. */

/* Kernel timing for roofline reporting: when enabled, CUDA events are recorded on the launch stream around the three
 * stages of every check call; artp_get_last_timing waits for the last call's kernels and returns
 * ms3[0..2] = classify (thread/item), box stages (warp stage + reach-box stages), plane-grouping block stage, in ms. */
int artp_set_timing(artp_handle* h, int enable);
int artp_get_last_timing(artp_handle* h, float* ms3);
/* Per-stage form: ms5 = classify, big-tile queue (torso boxes), reach-box queue (warp per box), reach-box queue (8-lane
 * groups), plane grouping. */
int artp_get_last_stage_timing(artp_handle* h, float* ms5);

/* Test hook: 0 = normal (classify -> warp stage -> grouping stage for deferred boxes),
 *            1 = send every in-map box through the exact block-level grouping kernel. */
int artp_set_mode(artp_handle* h, int mode);

/* ---- processors::Basic::setMaskedElevationAndTraversability (art_planner/src/map/processors/basic.cpp:42-106) ------
 * The producer of `elevation_masked` on the device: traversability threshold (+ "observed" masking), hole closing,
 * drop / wall masks, safety-margin erosion, small-patch removal -- grey-scale morphology with OpenCV's circular
 * structuring element (art_planner/src/utils.cpp:106-209) as exact min / max filters -- then
 * elevation_masked = traversable ? elevation : -inf. Inputs are the INPAINTED layers (basic.cpp:44-45: TELEA inpainting
 * is a sequential fast-marching method and stays with the caller); HOST pointers, grid_map layout; `observed` may be NULL
 * when !unknown_space_untraversable. Outputs: elevation_masked and (nullable) "traversability_thresholded". */
typedef struct artp_basic_params {
  float  traversability_thres;                        /* params.h:23 */
  int    unknown_space_untraversable;                 /* params.h:26 */
  double foothold_margin, foothold_margin_max_hole_size, foothold_margin_max_drop,
         foothold_margin_max_drop_search_radius, foothold_margin_min_step, foothold_size;   /* params.h:28-35 */
} artp_basic_params;
int artp_process_basic(artp_handle* h, const float* elevation, const float* traversability, const float* observed, int rows,
                       int cols, double res, const artp_basic_params* bp, float* elevation_masked, float* traversability_thresholded);
/* Test hook: the size x size structuring element of getCircularKernel(size) (utils.cpp:106-111) as 0/1 bytes; returns its
 * edge length (3 for size <= 0: OpenCV's default box). */
int artp_debug_circular_kernel(int size, uint8_t* out);

/* ---- learned motion cost (MotionCostFunc, objectives/motion_cost_objective.h:22-23) ------------------------------
 * Weights: ONE flat fp32 blob in the layer order of the reference's `network` module (network_light.py:9-63):
 * init_conv1..5, init_flatten, tar0_conv1, out0_conv1, out1_conv1..3 -- each conv.weight [Cout][Cin][kh][kw] followed by
 * its BatchNorm weight, bias, running_mean, running_var -- then out2_conv1..3 as conv.weight followed by conv.bias.
 * artp_cost_weights_size() floats in total (583 767 parameters + BN buffers). */
size_t artp_cost_weights_size(void);
int artp_set_cost_weights(artp_handle* h, const float* blob, size_t n_floats);
/* CostPredictor.updateFeatures (predictor.py:28-36): run the CNN trunk over the `elevation` layer of the current map
 * (orientation as cost_query_server.py:74). Call after artp_set_map whenever the map changed. */
int artp_update_features(artp_handle* h);
/* GPUCostQueryServer.handle_cost_query_no_update (cost_query_server.py:120-141) = CostQuery.__call__: edges n x 6 floats
 * [target_x, target_y, target_yaw, start_x, start_y, start_yaw] in the map frame -> cost3 n x 3 floats
 * (energy, time, risk = 1 - p_success). HOST buffers. */
int artp_motion_cost(artp_handle* h, const float* edges, size_t n, float* cost3);
int artp_motion_cost_device(artp_handle* h, const float* d_edges, size_t n, float* d_cost3, void* stream);
/* PRMMotionCostMaintainer::updateEdges / computeCostForVertexEdges (prm_motion_cost.cpp:27-128) for n graph edges
 * (source vertex state s_start = v1, target vertex state s_target = v2): the [n x 6] float edge matrix
 * [tx, ty, tyaw, sx, sy, syaw] with getYawFromSO3 (utils.h:80-88) ... */
int artp_edge_matrix_from_states(const double* s_start, const double* s_target, size_t n, float* edges);
/* ... and the whole batch in one call: edge matrix -> cost query -> isFeasible / getCost per row. cost[i] = +inf for
 * infeasible (too risky) edges exactly like updateEdges (:56-59); cost3 (nullable): the raw (energy, time, risk) rows. */
int artp_motion_cost_states(artp_handle* h, const double* s_start, const double* s_target, size_t n, double* cost,
                            uint8_t* feasible, float* cost3);
/* MotionCostObjective::getCost / isFeasible (motion_cost_objective.h:54-66) on host arrays:
 * cost[i] = w_e*E + w_t*T + w_r*R, feasible[i] = R <= risk_threshold (weights / threshold from artp_params). */
int artp_combine_cost(artp_handle* h, const float* cost3, size_t n, double* cost, uint8_t* feasible);
/* Test hooks: feature map copy-out ([Hf][Wf][48] fp32, channels last), kernel selection (bit 0: CUDA-core fp32
 * reference for the 15x15 layer instead of tcgen05; bit 1: set the smem-descriptor base_offset, a known-wrong variant kept for the record; bits 2-3: 15x15 layer variant, 0 = two-phase (default), 1 = single phase, 2 = single phase with CTA-pair weight multicast), trunk timings
 * ms3 = (3x3 stack, 15x15 layer, whole trunk) of the last artp_update_features. */
int artp_get_features(artp_handle* h, float* out, size_t n_floats, int* hf, int* wf);
int artp_set_cnn_mode(artp_handle* h, int mode);
int artp_get_cnn_timing(artp_handle* h, float* ms3);

/* ---- processors::computeChange + LazyPRMStarMinUpdateMaintainer::update (roadmap reuse across replans) -----------
 * grid_map_core is not in the reference tree, so its SubmapGeometry, index <-> position maps and LineIterator are used in
 * the written form DESIGN.md section 4.6 gives (buffer start index (0,0)); results are exact (float compares and integer
 * grid walks). */
typedef struct artp_grid {            /* one map's geometry + the two layers computeChange reads */
  const float* elevation;             /* grid_map layout, rows x cols column-major; NaN / inf allowed */
  const float* traversability_thresholded;
  int rows, cols; double res, cx, cy;
} artp_grid;
/* computeChange(map_new, map_old, height_change_for_update) (change.cpp:9-51): `updated` of the new map is 1 except over
 * the overlap of SubmapGeometry(new, old.position, old.length) and SubmapGeometry(old, new.position, new.length), where a
 * cell is 0 unless |e_new - e_old| > thr or t_old - t_new > 0.5 (float; NaN compares false). Either submap failing
 * leaves all ones. The layer stays on the handle, one bit per cell, with the new map's geometry, until the next
 * artp_compute_change; `updated` (nullable) receives it as floats (exact 0 / 1) in the new map's layout. HOST layers. */
int artp_compute_change(artp_handle* h, const artp_grid* map_new, const artp_grid* map_old,
                        float height_change_for_update, float* updated);
/* Same with DEVICE layers on `stream`, asynchronous; d_updated nullable. */
int artp_compute_change_device(artp_handle* h, const artp_grid* map_new, const artp_grid* map_old,
                               float height_change_for_update, float* d_updated, void* stream);
/* Against the last change layer (ARTP_E_NOMAP before the first artp_compute_change; artp_set_map is not needed):
 * vertex_flags[v]: 0 keep, 1 updated (-> VALIDITY_UNKNOWN), 2 outside the new map (removeOutdatedVertices), from x, y of
 * vertex_states (nv x 7 doubles, x y z qx qy qz qw);
 * edge_flags[e] for edges[e] = (source, target) vertex indices: 0, 1 a cell of grid_map's LineIterator from source to
 * target is updated, 2 an endpoint is outside (the edge goes with its vertex and is never walked).
 * Every edge index must be < nv: the host entry returns ARTP_E_INVALID before launching anything; the device entry
 * fails closed (flag 1) and raises the sticky error that artp_poll_error reports as ARTP_E_INVALID. */
int artp_roadmap_updates(artp_handle* h, const double* vertex_states, size_t nv,
                         const uint32_t* edges, size_t ne, uint8_t* vertex_flags, uint8_t* edge_flags);
int artp_roadmap_updates_device(artp_handle* h, const double* d_vertex_states, size_t nv, const uint32_t* d_edges,
                                size_t ne, uint8_t* d_vertex_flags, uint8_t* d_edge_flags, void* stream);

/* Version string of the library / kernel image ("artp <ver> sm_100a"). */
const char* artp_version(void);

#ifdef __cplusplus
}
#endif
#endif
