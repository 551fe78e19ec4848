/*
 * kompass_b200.h — C-ABI of the B200-native (sm_100a) DWA / local-mapper / critical-zone hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, opaque handles, int status codes. Every
 * entry point names the reference interface it replaces ("ref:" paths are relative to
 * /root/reference/src/kompass_cpp/kompass_cpp/). The reference-side bindings a maintainer would
 * add are shown in INTEGRATION.md. There is NO CPU fallback: every call fails with KC_ERR_CUDA if
 * no CUDA device is usable.
 *
 * Threading: handles are not thread-safe; distinct handles may be driven from distinct threads.
 * Each handle owns one CUDA stream, its device buffers and pinned staging memory. Calls are
 * synchronous: they return when results are in host memory. Output pointers returned inside
 * result structs are library-owned pinned host buffers, valid until the next call on that handle.
 */
#ifndef KOMPASS_B200_H
#define KOMPASS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes (C++ wrapper maps: INVALID_ARG -> std::invalid_argument, others ->
 *      std::runtime_error, OUT_OF_RANGE -> std::out_of_range; "no admissible trajectory" is NOT
 *      an error: found = 0, ref: include/controllers/dwa.h:219-221) ---- */
enum {
  KC_OK = 0,
  KC_ERR_INVALID_ARG = 1,
  KC_ERR_CUDA = 2,
  KC_ERR_OOM = 3,
  KC_ERR_UNSUPPORTED = 4,
  KC_ERR_OUT_OF_RANGE = 5
};

/* ref: include/datatypes/control.h:14 ControlType */
enum { KC_ACKERMANN = 0, KC_DIFFERENTIAL_DRIVE = 1, KC_OMNI = 2 };
/* ref: include/utils/collision_check.h:25 CollisionChecker::ShapeType */
enum { KC_CYLINDER = 0, KC_BOX = 1, KC_SPHERE = 2 };
/* ref: include/mapping/local_mapper.h:9 OccupancyType */
enum { KC_UNEXPLORED = -1, KC_EMPTY = 0, KC_OCCUPIED = 100 };
/* ref: include/utils/pointcloud.h:37-46 PointFieldType */
enum {
  KC_INT8 = 1, KC_UINT8 = 2, KC_INT16 = 3, KC_UINT16 = 4,
  KC_INT32 = 5, KC_UINT32 = 6, KC_FLOAT32 = 7, KC_FLOAT64 = 8
};

/* Text of the last error raised on the calling thread ("" if none). */
const char *kc_last_error(void);
/* ref: src/utils/gpu_check.cpp:7-22 getAvailableAccelerators(): newline separated device names;
 * returns the number of CUDA devices (0 when none). */
int32_t kc_available_accelerators(char *buf, int32_t buf_len);
/* Library / build identification: "kompass_b200 <ver> sm_100a". */
const char *kc_version(void);

/* =============================================================================================
 * DWA planner = TrajectorySampler + CollisionChecker + CostEvaluator + best-trajectory selection.
 * ref: include/controllers/dwa.h:24-41 (ctor args), include/utils/trajectory_sampler.h:22-91,
 *      include/utils/cost_evaluator.h:22-93
 * ========================================================================================== */
typedef struct kc_planner kc_planner;

typedef struct kc_planner_config {
  int32_t control_type;          /* KC_ACKERMANN / KC_DIFFERENTIAL_DRIVE / KC_OMNI */
  double time_step;              /* "time_step" */
  double prediction_horizon;     /* "prediction_horizon" [s] (upper bound for adaptation) */
  double control_horizon;        /* "control_horizon" [s] */
  int32_t max_linear_samples;    /* "max_linear_samples" */
  int32_t max_angular_samples;   /* "max_angular_samples" */
  /* ref: include/datatypes/control.h:181-232 ControlLimitsParams: maxVel, maxAcc, maxDec */
  double vx_max, vx_acc, vx_dec;
  double vy_max, vy_acc, vy_dec;
  double omega_max, omega_acc, omega_dec;
  int32_t robot_shape;           /* KC_CYLINDER {r,h} / KC_BOX {x,y,z} / KC_SPHERE {r} */
  float robot_dims[3];
  float sensor_position[3];      /* sensor_position_body */
  float sensor_rotation[4];      /* sensor_rotation_body as Eigen coeffs (x,y,z,w) */
  double octree_resolution;      /* "octree_map_resolution" */
  int32_t drop_samples;          /* "drop_samples" */
  int64_t num_ctrl_points;       /* <0: derive control_horizon/time_step (trajectory_sampler.cpp:88) */
  /* ref: cost_evaluator.h:22-50 TrajectoryCostsWeights */
  double w_path, w_goal, w_obstacles, w_smooth, w_jerk;
  float max_local_range;         /* DWA::maxLocalRange_, default 10 (dwa.h:236) */
  int32_t max_num_threads;       /* accepted for signature parity, ignored */
} kc_planner_config;

/* One control-cycle result. ref: include/datatypes/trajectory.h:611-618 TrajSearchResult */
typedef struct kc_cycle_result {
  int32_t found;        /* isTrajFound */
  float cost;           /* trajCost (FLT_MAX when !found after evaluation, 0 when no sample) */
  int32_t slot;         /* enumeration index of the winner among all sampled velocity slots */
  int32_t n_points;     /* numPointsPerTrajectory of this cycle (P) */
  int32_t n_slots;      /* velocity slots enumerated this cycle */
  int32_t n_admissible; /* samples_->size(): collision-free samples */
  const float *vx, *vy, *omega; /* winner velocities [P-1] */
  const float *x, *y;           /* winner path [P] */
} kc_cycle_result;

/* Batch of admissible samples. ref: include/datatypes/trajectory.h:506-603 TrajectorySamples2D */
typedef struct kc_samples {
  int32_t count;    /* size() */
  int32_t n_points; /* P */
  const float *vx, *vy, *omega; /* row-major [count x (P-1)] */
  const float *x, *y;           /* row-major [count x P] */
  const int32_t *slots;         /* enumeration index of each row */
} kc_samples;

int32_t kc_planner_create(const kc_planner_config *cfg, kc_planner **out);
void kc_planner_destroy(kc_planner *p);

/* ref: CostEvaluator::updateCostWeights (cost_evaluator.h:231) */
int32_t kc_planner_set_weights(kc_planner *p, double w_path, double w_goal, double w_obstacles,
                               double w_smooth, double w_jerk);
/* ref: DWA::resetOctreeResolution (dwa.cpp:139-141) */
int32_t kc_planner_set_octree_resolution(kc_planner *p, double resolution);
/* ref: TrajectorySampler::setSampleDroppingMode (trajectory_sampler.cpp:98-100) */
int32_t kc_planner_set_drop_samples(kc_planner *p, int32_t drop);
/* ref: DWA::setSensorMaxRange (dwa.cpp:143-145) */
int32_t kc_planner_set_max_range(kc_planner *p, float max_range);
float kc_planner_get_max_range(const kc_planner *p);
/* velocity slots enumerated by the last cycle / sampler call on this handle */
int32_t kc_planner_num_slots_last(const kc_planner *p);
/* ref: TrajectorySampler::setPredictionHorizon (trajectory_sampler.cpp:316-326); clamps to
 * [2*time_step, base horizon]; returns the resulting points-per-trajectory through *n_points. */
int32_t kc_planner_set_prediction_horizon(kc_planner *p, double horizon, int32_t *n_points);
/* ref: trajectory.h:32-51 getNumTrajectories / getNumPointsPerTrajectory */
int32_t kc_planner_num_trajectories(const kc_planner *p);
int32_t kc_planner_num_points(const kc_planner *p);

/* Upload the interpolated reference path (Path::X_/Y_/accumulated_path_length_, ref:
 * include/datatypes/path.h:287-297) once; cycles then name the tracked segment by (start,count)
 * exactly as Path::View does (path.h:55-61). total_length = Path::totalPathLength(). */
int32_t kc_planner_set_path(kc_planner *p, const float *X, const float *Y, const float *acc,
                            int32_t n, float total_length);

/* Full DWA cycle = DWA::findBestPath (dwa.h:183-230) from generateTrajectories on:
 * sample + rollout + collision + setPointScan + getMinTrajectoryCost.
 * vel = {vx, vy, omega} (Velocity2D), pose = {x, y, yaw} (Path::State).
 * Laser-scan overload: ranges/angles as in Control::LaserScan (control.h:237-243).
 * Point-cloud overload: xyz = n packed Path::Point (Eigen::Vector3f), i.e. 3 floats per point. */
int32_t kc_planner_cycle_scan(kc_planner *p, const double vel[3], const double pose[3],
                              const double *ranges, const double *angles, int32_t n,
                              int32_t seg_start, int32_t seg_count, kc_cycle_result *out);
int32_t kc_planner_cycle_cloud(kc_planner *p, const double vel[3], const double pose[3],
                               const float *xyz, int32_t n, int32_t seg_start, int32_t seg_count,
                               kc_cycle_result *out);
/* Per-slot total cost (FLT_MAX for inadmissible slots) and admissible flags of the last cycle
 * (parity/debug surface; costs and flags are [n_slots]). Either pointer may be NULL. */
int32_t kc_planner_fetch_costs(kc_planner *p, float *costs, uint8_t *admissible);
/* The cycle finds the argmin by branch and bound: a slot whose lower bound (goal + path cost + the
 * obstacle term bounded from the per-cell distance table) exceeds another slot's upper bound cannot
 * win, and its exact obstacle search is skipped. pruned[i] = 1 marks those slots: their entry in
 * `costs` is that lower bound, not the total (tuning key 7 = 0 evaluates every slot exactly; by
 * default cycles with fewer than 2048 slots are evaluated exactly too). The winner, its cost and its
 * rows never depend on the setting. */
int32_t kc_planner_fetch_pruned(kc_planner *p, uint8_t *pruned);

/* TrajectorySampler::generateTrajectories (trajectory_sampler.h:114-121): admissible samples in
 * enumeration order, copied to pinned host memory. */
int32_t kc_sampler_generate_scan(kc_planner *p, const double vel[3], const double pose[3],
                                 const double *ranges, const double *angles, int32_t n,
                                 kc_samples *out);
int32_t kc_sampler_generate_cloud(kc_planner *p, const double vel[3], const double pose[3],
                                  const float *xyz, int32_t n, kc_samples *out);

/* CostEvaluator::setPointScan (cost_evaluator.h:174-223). n = 0 clears the obstacle list. */
int32_t kc_cost_set_points_scan(kc_planner *p, const double *ranges, const double *angles,
                                int32_t n, const double pose[3], float max_sensor_range,
                                float max_obstacle_cost_range_multiple);
int32_t kc_cost_set_points_cloud(kc_planner *p, const float *xyz, int32_t n, const double pose[3],
                                 float max_sensor_range, float max_obstacle_cost_range_multiple);
/* CostEvaluator::getMinTrajectoryCost (cost_evaluator.h:139-142) on caller-provided samples
 * (row-major host arrays as in TrajectorySamples2D). custom: optional host-evaluated callback terms,
 * row-major [n_traj x n_custom] doubles holding weight_k * custom_cost_k(trajectory, path); each is
 * added as `total_cost (float) += term (double)` in registration order, exactly as
 * cost_evaluator.cpp:96-100 does (n_custom = 0: none);
 * costs_out: optional per-trajectory totals [n_traj]. */
int32_t kc_cost_evaluate(kc_planner *p, int32_t n_traj, int32_t n_points, const float *vx,
                         const float *vy, const float *omega, const float *x, const float *y,
                         int32_t seg_start, int32_t seg_count, const double *custom,
                         int32_t n_custom, float *costs_out, kc_cycle_result *out);

/* ---- device-resident replay (measurement only; inputs already in HBM) ----
 * A bank of point clouds is uploaded once; kc_planner_replay enqueues n_cycles full cycles
 * back-to-back on the handle's stream, cycle i using bank slot (first_slot + i) % n_slots, with
 * no host synchronisation in between, and reports CUDA-event times measured on that stream:
 * total_ms over all cycles and eval_ms = summed duration of the rollout+collision+cost kernel. */
int32_t kc_planner_bank_alloc(kc_planner *p, int32_t n_slots, int32_t max_points);
int32_t kc_planner_bank_upload(kc_planner *p, int32_t slot, const float *xyz, int32_t n);
int32_t kc_planner_replay(kc_planner *p, int32_t first_slot, int32_t n_cycles, const double vel[3],
                          const double pose[3], int32_t seg_start, int32_t seg_count,
                          float *total_ms, float *eval_ms, kc_cycle_result *last);
/* Kernel launches issued by this handle since creation (bench.py's gpu_launches claim). */
int64_t kc_planner_launch_count(const kc_planner *p);
/* Page-locked host memory (optional): sensor arrays that live in it (or in any cudaHostAlloc /
 * cudaHostRegister-ed memory) are DMA-ed straight from the caller's buffer by kc_planner_cycle_* /
 * kc_dwa_compute_*; ordinary pageable buffers are staged through the handle's own pinned buffer. */
void *kc_pinned_alloc(size_t bytes);
void kc_pinned_free(void *ptr);
/* Test/diagnostic hooks (no reference counterpart). Tuning keys: 0 = candidate-pool capacity per
 * robot (0 forces the generic exact obstacle search for every cell; results are identical by
 * construction and the parity tests run both ways); 1 = replay each cycle's launch set as a cached
 * CUDA graph (1, default) or as plain launches (0); 2 = a page-locked caller cloud is read in place
 * over PCIe by the one kernel that consumes it (1, default) or DMA-ed into HBM first (0); 3 = the
 * winner record is written straight into the handle's pinned result buffer (1, default) or copied
 * back with a D2H memcpy (0); 4 = developer timeline (see kc_planner_debug_timeline); 5 = candidate
 * lists are built only for grid cells inside the analytic reach set of the velocity window (1,
 * default; queries outside it take the generic exact search, results identical) or for the whole
 * query window (0); 6 = retired, accepted and ignored; 7 =
 * branch and bound over the slots: 0 = every slot evaluated exactly, 1 = when the cycle has at least
 * 2048 velocity slots (default), 2 = always; 8 = the host watches the mapped result record for the
 * cycle's sequence number (1, default) instead of waiting on the stream (0); 9 = the kernels that
 * follow the bounds stage are programmatic dependent launches (1, default; environment KC_PDL=0
 * turns the default off) or plain stream-ordered ones (0); 10 = policy for query cells whose search
 * disc holds thousands of points (a dense cluster, a wall seen by a depth camera): -1 (default) = such
 * cells get only their exact centre distance, from a CTA-cooperative kernel that is launched while the
 * previous cycle reported such cells, and their rare exact queries run a warp-cooperative search; N > 0 =
 * the same with threshold N points and the kernel always launched; 0 = every cell builds its list with
 * its own warp (results identical in all three); 11 = per-cell candidate lists: 1 (default) = always
 * built, -1 = only when every slot is evaluated exactly, 0 = never (exact queries then search their
 * own disc; results identical, slower when the bounds leave hundreds of survivors); 12 = robots per
 * launch set of a batched sweep (1..64; the sweep starts with chunks of 8, 16, 32 robots so that little
 * of the cloud upload runs un-overlapped); 13 = number of slots that survive the bound stage up to
 * which the exact stage spreads (slot, point) pairs over the whole grid in batches instead of handing
 * whole slots to warps (default 2048; 0 = always by slot; results identical). Stats of the last
 * single-robot cycle:
 * out[0] pool entries used, [1] query-window cells, [2] cells with a candidate list,
 * [3] cells marked for the generic search, [4] longest list, [5] obstacle points kept by the cull,
 * [6] tracked-segment candidate entries used, [7] longest tracked-segment list. */
int32_t kc_planner_set_tuning(kc_planner *p, int32_t key, int64_t value);
/* Verification / roofline hook (never on the control path): the obstacle-distance cost of every
 * velocity slot of the LAST kc_planner_cycle_* call, by brute force exactly as
 * TrajectoryPath::minDist2D + obstaclesDistCostFunc are written (include/datatypes/trajectory.h:
 * 218-235, src/utils/cost_evaluator.cpp:179-184): every admissible trajectory point against EVERY
 * sensor point, no cull, no grid. costs [n_slots] (FLT_MAX for inadmissible slots). pass1_ms = CUDA-
 * event time of the FP32 pass (N*P*M pair evaluations, 6 FLOP each as SURVEY 8(d) counts them);
 * pair_evaluations = N*P*M. total_ms is reserved (0). Any of the three may be NULL. */
int32_t kc_planner_bruteforce_obstacle_costs(kc_planner *p, float *costs, float *pass1_ms,
                                             float *total_ms, double *pair_evaluations);
int32_t kc_planner_debug_stats(kc_planner *p, int64_t out[8]);
/* Developer time stamps inside k_cost_eval (only meaningful in a library built with
 * -DKC_DBG_STAMPS; tools/stamps_dev.py): reset = 1 arms them, reset = 0 reads them into out[0..7]
 * (nanoseconds after the first CTA's start). */
int32_t kc_planner_debug_stamps(kc_planner *p, int32_t reset, int64_t out[8]);
/* Developer timeline (tuning key 4 = 1: every kernel of a cycle is bracketed by CUDA events on the
 * stream it runs on, plain launches): kernel names and (start, end) in microseconds after the cycle's
 * first event; returns the number of kernels written (<= cap). */
int32_t kc_planner_debug_timeline(kc_planner *p, const char **names, float *start_us, float *end_us,
                                  int32_t cap);

/* =============================================================================================
 * DWA controller (SURVEY section 8 row f1): the reference's Follower/DWA layer around the planner.
 * Replaces Kompass::Control::DWA as the Python bindings see it (bindings_control.cpp:221-273) plus
 * the Follower/Controller methods it inherits (:66-106):
 *   setCurrentPath       src/controllers/follower.cpp:81-107 (Path::interpolate LINEAR + segment,
 *                        src/datatypes/path.cpp:167-330)
 *   setCurrentState      src/controllers/dwa.cpp:152-155
 *   compute*             include/controllers/dwa.h:113-139,183-230: determineTarget
 *                        (follower.cpp:262-304) -> adaptPredictionHorizonToCurvature
 *                        (dwa.cpp:157-206) -> findTrackedPathSegment (dwa.cpp:208-233) -> one
 *                        planner cycle on the GPU
 *   isGoalReached        follower.cpp:111-145
 * The handle owns a kc_planner (kc_dwa_planner) for the setters above (weights, resolution, range).
 * ========================================================================================== */
typedef struct kc_dwa kc_dwa;
typedef struct kc_follower_params { /* ref: follower.h:24-75 FollowerParameters */
  double max_point_interpolation_distance; /* 0.01 */
  double lookahead_distance;               /* 1.0  */
  double goal_dist_tolerance;              /* 0.1  */
  double path_segment_length;              /* 1.0  */
  double goal_orientation_tolerance;       /* 0.1  */
  double loosing_goal_distance;            /* 0.5  */
  double curvature_horizon_tolerance;      /* 1.5  */
} kc_follower_params;
typedef struct kc_dwa_info { /* what the last compute call tracked (Follower::Target + the view) */
  int32_t closest_index, segment_index, seg_start, seg_count, n_points, _pad;
  double segment_position, crosstrack_error, heading_error, horizon;
  double target_x, target_y, target_yaw;
} kc_dwa_info;
void kc_follower_params_default(kc_follower_params *p);
/* Path::interpolate (LINEAR, path.cpp:167-288) + Path::segment (path.cpp:290-330) on the host; no
 * device needed. Arrays of capacity `cap`; acc[i] = Path::getDistanceAtIndex(i). */
int32_t kc_path_prepare(const float *x, const float *y, int32_t n, int32_t interpolate,
                        double max_point_interpolation_distance, double path_segment_length,
                        int64_t max_points_per_segment, int32_t cap, float *X, float *Y, float *acc,
                        float *curvature, int32_t *seg_starts, int32_t *n_out, int32_t *n_segments,
                        float *total_length);
int32_t kc_dwa_create(const kc_planner_config *cfg, const kc_follower_params *follower /* NULL: defaults */,
                      kc_dwa **out);
void kc_dwa_destroy(kc_dwa *d);
kc_planner *kc_dwa_planner(kc_dwa *d);
int32_t kc_dwa_set_current_path(kc_dwa *d, const float *x, const float *y, int32_t n, int32_t interpolate);
int32_t kc_dwa_clear_current_path(kc_dwa *d);
int32_t kc_dwa_set_current_state(kc_dwa *d, double x, double y, double yaw, double speed);
int32_t kc_dwa_set_control_limits(kc_dwa *d, double vx_max, double vy_max, double omega_max);
int32_t kc_dwa_is_goal_reached(kc_dwa *d, int32_t *reached);
int32_t kc_dwa_has_path(const kc_dwa *d);
int32_t kc_dwa_get_path(const kc_dwa *d, const float **X, const float **Y, const float **curvature,
                        int32_t *n, int32_t *n_segments, float *total_length);
int32_t kc_dwa_get_command(const kc_dwa *d, double cmd[3]);
/* Custom trajectory costs. ref: DWA::addCustomCost (src/controllers/dwa.cpp:147-150) ->
 * CostEvaluator::addCustomCost (include/utils/cost_evaluator.h:150-154); CustomCostFunction =
 * double(const Trajectory2D&, const Path::Path&) (cost_evaluator.h:97-98). The callback sees one
 * admissible trajectory and the whole current reference path; it runs on the calling thread during
 * kc_dwa_compute_*. While any callback is registered a cycle runs the reference's own three steps
 * (generateTrajectories -> callbacks on the host -> setPointScan + getMinTrajectoryCost with the
 * terms added as `float += weight * value` in registration order) instead of the fused launch set. */
typedef struct kc_trajectory_view {
  int32_t n_points;             /* P */
  const float *vx, *vy, *omega; /* [P-1] */
  const float *x, *y;           /* [P] */
} kc_trajectory_view;
typedef struct kc_path_view {
  int32_t n;
  const float *X, *Y; /* the current (interpolated) reference path */
  const float *acc;   /* acc[i] = Path::getDistanceAtIndex(i) */
  float total_length; /* Path::totalPathLength() */
} kc_path_view;
typedef double (*kc_custom_cost_fn)(const kc_trajectory_view *trajectory, const kc_path_view *reference_path,
                                    void *user);
int32_t kc_dwa_add_custom_cost(kc_dwa *d, double weight, kc_custom_cost_fn fn, void *user);
int32_t kc_dwa_clear_custom_costs(kc_dwa *d);
/* ref: DWA::debugVelocitySearch<T> (include/controllers/dwa.h:147-165): determineTarget, set the
 * sampler's dropping mode (it stays set), generateTrajectories; the samples are kept by the handle.
 * `out` may be NULL. ref: DWA::getDebuggingSamples / getDebuggingSamplesPure
 * (src/controllers/dwa.cpp:235-250); KC_ERR_INVALID_ARG "No debugging samples are available" before
 * the first search. The arrays stay valid until the next debug search on this handle. */
int32_t kc_dwa_debug_velocity_search_scan(kc_dwa *d, const double vel[3], const double *ranges,
                                          const double *angles, int32_t n, int32_t drop_samples,
                                          kc_samples *out);
int32_t kc_dwa_debug_velocity_search_cloud(kc_dwa *d, const double vel[3], const float *xyz, int32_t n,
                                           int32_t drop_samples, kc_samples *out);
int32_t kc_dwa_get_debugging_samples(const kc_dwa *d, kc_samples *out);
/* out->* rows stay valid until the next call on this handle; info may be NULL */
int32_t kc_dwa_compute_scan(kc_dwa *d, const double vel[3], const double *ranges, const double *angles,
                            int32_t n, kc_cycle_result *out, kc_dwa_info *info);
int32_t kc_dwa_compute_cloud(kc_dwa *d, const double vel[3], const float *xyz, int32_t n,
                             kc_cycle_result *out, kc_dwa_info *info);

/* =============================================================================================
 * Stand-alone collision checker (SURVEY section 8 row f4). Replaces Kompass::CollisionChecker
 * (include/utils/collision_check.h:23-180, src/utils/collision_check.cpp:17-246) for its users
 * outside the DWA cycle: PurePursuit's avoidance rollouts (src/controllers/pure_pursuit.cpp:154-155),
 * OMPL state validity (src/planning/ompl.cpp:95-97) and TrajectorySampler::checkStatesFeasibility
 * (src/utils/trajectory_sampler.cpp:378-408). Same occupied-voxel model and robot-vs-voxel test as
 * the DWA rollout kernel (FCL 0.7 / octomap restated, see DESIGN.md section 2). Any sensor mount whose
 * sensor_rotation is a rotation (unit quaternion within 1e-3) is accepted: upright and upside-down mounts
 * keep the voxel cubes axis-aligned with the robot solid (2-D column test); pitched / rolled mounts turn
 * them into oriented boxes (sphere / box / cylinder against an oriented cube). getMinDistance (FCL
 * distance query, unused by the reference's own callers) is not provided.
 * ========================================================================================== */
typedef struct kc_collision kc_collision;
typedef struct kc_collision_config { /* CollisionChecker ctor, collision_check.h:45-49 */
  int32_t robot_shape;       /* KC_CYLINDER {r,h} / KC_BOX {x,y,z} / KC_SPHERE {r} */
  float robot_dims[3];
  float sensor_position[3];  /* sensor_position_body */
  float sensor_rotation[4];  /* sensor_rotation_body, Eigen coeffs (x,y,z,w) */
  double octree_resolution;  /* default 0.01 in the reference */
} kc_collision_config;
int32_t kc_collision_create(const kc_collision_config *cfg, kc_collision **out);
void kc_collision_destroy(kc_collision *c);
/* resetOctreeResolution (collision_check.cpp:70-75); applies from the next sensor update */
int32_t kc_collision_reset_octree_resolution(kc_collision *c, double resolution);
float kc_collision_get_radius(const kc_collision *c); /* getRadius */
/* updateState(x, y, yaw) / updateState(Path::State) (collision_check.cpp:125-147) */
int32_t kc_collision_update_state(kc_collision *c, double x, double y, double yaw);
/* updateSensorData<LaserScan> / <std::vector<Path::Point>>(data, global_frame)
 * (collision_check.h:91-136): the sensor-to-world transform is fixed here from the CURRENT state
 * (scan, or cloud with global_frame = 0); n = 0 clears the octree */
int32_t kc_collision_update_scan(kc_collision *c, const double *ranges, const double *angles, int32_t n);
int32_t kc_collision_update_cloud(kc_collision *c, const float *xyz, int32_t n, int32_t global_frame);
/* checkCollisions() at the current state (collision_check.cpp:149-162) */
int32_t kc_collision_check(kc_collision *c, int32_t *collides);
/* checkCollisions(Path::State) (collision_check.cpp:225-246) for n states at once: states = [n x 3]
 * doubles (x, y, yaw); collides [n] (may be NULL); *any = 1 if some state collides (may be NULL) =
 * TrajectorySampler::checkStatesFeasibility */
int32_t kc_collision_check_states(kc_collision *c, const double *states, int32_t n, uint8_t *collides,
                                  int32_t *any);

/* =============================================================================================
 * Batched multi-robot sweep: R independent robots (own velocity, pose, cloud), one launch set.
 * north_star config 5. All robots share the planner configuration and reference path.
 * vel/pose: [R x 3] doubles; xyz: robot r's cloud at xyz + 3*offsets[r], counts[r] points.
 * results: [R]. Winner rows are not returned (index + cost only, the "final result gather").
 * ========================================================================================== */
typedef struct kc_batch_result {
  int32_t found;
  float cost;
  int32_t slot;
  int32_t n_admissible;
  int32_t n_slots; /* velocity slots this robot enumerated (its share of the trajectory-steps) */
} kc_batch_result;
int32_t kc_planner_batch_cloud(kc_planner *p, int32_t n_robots, const double *vel,
                               const double *pose, const float *xyz, const int64_t *offsets,
                               const int32_t *counts, int32_t seg_start, int32_t seg_count,
                               kc_batch_result *results);
/* device-resident replay of the batch (inputs uploaded by the previous kc_planner_batch_cloud) */
int32_t kc_planner_batch_replay(kc_planner *p, int32_t n_iters, float *total_ms,
                                kc_batch_result *results);

/* =============================================================================================
 * Multi-robot DWA controller: R robots, each with its own reference path, state, control limits
 * and sensor data, stepped together in one batched launch set per chunk of robots. For every robot
 * r a step returns exactly what a kc_dwa handle with the same configuration, path, state and
 * sensor data returns from kc_dwa_compute_*: found, slot, cost bits, n_admissible, n_slots, P, the
 * winner rows, every kc_dwa_info field, the clamped command and the goal flag. The latest command
 * is kept when no trajectory is found. Custom cost callbacks and the debug velocity search stay
 * with kc_dwa.
 * Sensor data uses the layout of kc_planner_batch_cloud: robot r's cloud is xyz + 3*offsets[r]
 * (counts[r] points), its scan ranges + offsets[r] / angles + offsets[r] (counts[r] beams); robots
 * may share slices; page-locked clouds are DMA-ed directly. A step takes one sensor kind.
 * ========================================================================================== */
typedef struct kc_fleet kc_fleet;
typedef struct kc_fleet_result {
  int32_t found;
  float cost;
  int32_t slot, n_points, n_slots, n_admissible;
  double cmd[3]; /* command after this step, exactly what kc_dwa_get_command would return */
} kc_fleet_result;
/* follower: NULL = defaults. Fails with KC_ERR_CUDA without a device. */
int32_t kc_fleet_create(const kc_planner_config *cfg, const kc_follower_params *follower, int32_t n_robots,
                        kc_fleet **out);
void kc_fleet_destroy(kc_fleet *f);
/* the shared planner: weights, resolution, max range, drop mode, tuning keys */
kc_planner *kc_fleet_planner(kc_fleet *f);
/* Follower::setCurrentPath of one robot; its interpolated path goes to the device once, here */
int32_t kc_fleet_set_current_path(kc_fleet *f, int32_t robot, const float *x, const float *y, int32_t n,
                                  int32_t interpolate);
int32_t kc_fleet_clear_current_path(kc_fleet *f, int32_t robot);
/* states: [R x 4] doubles (x, y, yaw, speed) */
int32_t kc_fleet_set_current_states(kc_fleet *f, const double *states);
/* Controller limits of every robot (as kc_dwa_set_control_limits) */
int32_t kc_fleet_set_control_limits(kc_fleet *f, double vx_max, double vy_max, double omega_max);
/* one step of every robot. vel: [R x 3]; results: [R]; info: [R] or NULL. A robot without a path
 * fails the call with KC_ERR_INVALID_ARG naming it. */
int32_t kc_fleet_compute_cloud(kc_fleet *f, const double *vel, const float *xyz, const int64_t *offsets,
                               const int32_t *counts, kc_fleet_result *results, kc_dwa_info *info);
int32_t kc_fleet_compute_scan(kc_fleet *f, const double *vel, const double *ranges, const double *angles,
                              const int64_t *offsets, const int32_t *counts, kc_fleet_result *results,
                              kc_dwa_info *info);
/* the winner record of one robot's last step (rows valid until the next call on the fleet) */
int32_t kc_fleet_get_trajectory(const kc_fleet *f, int32_t robot, kc_cycle_result *out);
/* Follower::isGoalReached of every robot: reached [R] */
int32_t kc_fleet_is_goal_reached(kc_fleet *f, int32_t *reached);

/* =============================================================================================
 * Local mapper. ref: include/mapping/local_mapper_gpu.h:12-147 (LocalMapperGPU ctor + 2
 * scanToGrid overloads); arithmetic follows the reference CPU LocalMapper::scanToGrid
 * (src/mapping/local_mapper.cpp:127-159,204-251), which is the parity target.
 * ========================================================================================== */
typedef struct kc_mapper kc_mapper;
typedef struct kc_mapper_config {
  int32_t grid_height, grid_width;
  float resolution;
  float laserscan_position[3];
  float laserscan_orientation;
  int32_t is_pointcloud;
  int32_t scan_size;
  float angle_step;   /* overridden by 2*pi/scan_size for point clouds (local_mapper.h:39-55) */
  float max_height, min_height, range_max;
  int32_t max_points_per_line; /* accepted, unused (rays are walked to their end point) */
} kc_mapper_config;
int32_t kc_mapper_create(const kc_mapper_config *cfg, kc_mapper **out);
void kc_mapper_destroy(kc_mapper *m);
/* grid_out: column-major int32 [H x W] (Eigen::MatrixXi layout: cell (i,j) at i + j*H). */
int32_t kc_mapper_scan_to_grid(kc_mapper *m, const double *angles, const double *ranges, int32_t n,
                               int32_t *grid_out);
int32_t kc_mapper_cloud_to_grid(kc_mapper *m, const int8_t *data, int64_t nbytes,
                                int32_t point_step, int32_t row_step, int32_t height, int32_t width,
                                float x_offset, float y_offset, float z_offset, int32_t *grid_out);
/* device-resident replay of the last scan (measurement only) */
int32_t kc_mapper_replay(kc_mapper *m, int32_t n_iters, float *total_ms);
/* Bayesian mapper (SURVEY section 8 row f2). ref: LocalMapper::scanToGridBaysian(angles, ranges)
 * (src/mapping/local_mapper.cpp:106-125,161-202,222-238), getPreviousGridInCurrentPose (:17-78) and
 * the Bayesian constructor's extra arguments (include/mapping/local_mapper.h:58-75; defaults of the
 * 13-argument constructor: prior 0.5, occupied 0.6, empty 0.4, range_sure 1.0, wall_size 0.2).
 * Serial-order semantics: the last ray crossing a cell decides its probability. prob_out and the
 * previous grid are column-major float [H x W] like Eigen::MatrixXf. */
int32_t kc_mapper_set_bayesian_params(kc_mapper *m, float p_prior, float p_occupied, float p_empty,
                                      float range_sure, float wall_size);
int32_t kc_mapper_scan_to_grid_bayesian(kc_mapper *m, const double *angles, const double *ranges,
                                        int32_t n, int32_t *grid_out, float *prob_out);
/* ref: LocalMapper::scanToGridBaysian(raw cloud) (src/mapping/local_mapper.cpp:253-264): bins the
 * cloud with the ANGLE-STEP overload of pointCloudToLaserScanFromRaw (include/utils/pointcloud.h:
 * 116-177) using the constructor's angle_step as given, then the scan overload. */
int32_t kc_mapper_cloud_to_grid_bayesian(kc_mapper *m, const int8_t *data, int64_t nbytes,
                                         int32_t point_step, int32_t row_step, int32_t height,
                                         int32_t width, float x_offset, float y_offset, float z_offset,
                                         int32_t *grid_out, float *prob_out);
int32_t kc_mapper_previous_grid_in_current_pose(kc_mapper *m, float pos_x, float pos_y,
                                                double orientation);
int32_t kc_mapper_get_previous_grid(kc_mapper *m, float *prob_out);
int32_t kc_mapper_set_previous_grid(kc_mapper *m, const float *prob);

/* ref: include/utils/pointcloud.h:205-259 pointCloudToLaserScanFromRaw (num_bins overload) */
int32_t kc_pointcloud_to_laserscan(const int8_t *data, int64_t nbytes, int32_t point_step,
                                   int32_t row_step, int32_t height, int32_t width, int32_t x_offset,
                                   int32_t y_offset, int32_t z_offset, double max_range,
                                   double min_z, double max_z, int32_t num_bins,
                                   double *ranges_out);

/* ref: include/utils/pointcloud.h:116-177 (angle_step overload): n = ceil(2 pi / angle_step) bins,
 * bin = int(angle / angle_step), angles_out[i] = i * angle_step; arrays of capacity `cap`. */
int32_t kc_pointcloud_to_laserscan_step(const int8_t *data, int64_t nbytes, int32_t point_step,
                                        int32_t row_step, int32_t height, int32_t width,
                                        int32_t x_offset, int32_t y_offset, int32_t z_offset,
                                        double max_range, double min_z, double max_z,
                                        double angle_step, int32_t cap, double *ranges_out,
                                        double *angles_out, int32_t *n_bins_out);

/* =============================================================================================
 * Critical zone checker. ref: include/utils/critical_zone_check_gpu.h:17-192
 * (CriticalZoneCheckerGPU ctor + 2 check overloads); arithmetic follows the CPU
 * CriticalZoneChecker (src/utils/critical_zone_check.cpp:13-131), the parity target.
 * ========================================================================================== */
typedef struct kc_critical_zone kc_critical_zone;
typedef struct kc_critical_zone_config {
  int32_t input_type;      /* 0 LASERSCAN, 1 POINTCLOUD (critical_zone_check.h:15-18) */
  int32_t robot_shape;
  float robot_dims[3];
  float sensor_position[3];
  float sensor_rotation[4]; /* (x,y,z,w), used un-normalised like the reference */
  float critical_angle;     /* degrees */
  float critical_distance;
  float slowdown_distance;
  float min_height, max_height, range_max;
  int32_t cloud_field_type; /* KC_FLOAT32 only (the CPU reference memcpy's floats) */
} kc_critical_zone_config;
int32_t kc_critical_zone_create(const kc_critical_zone_config *cfg, const double *angles,
                                int32_t n_angles, kc_critical_zone **out);
void kc_critical_zone_destroy(kc_critical_zone *z);
int32_t kc_critical_zone_check_scan(kc_critical_zone *z, const double *ranges, int32_t n,
                                    int32_t forward, float *factor_out);
int32_t kc_critical_zone_check_cloud(kc_critical_zone *z, const int8_t *data, int64_t nbytes,
                                     int32_t point_step, int32_t row_step, int32_t height,
                                     int32_t width, int32_t x_offset, int32_t y_offset,
                                     int32_t z_offset, int32_t forward, float *factor_out);
int32_t kc_critical_zone_replay(kc_critical_zone *z, int32_t n_iters, float *total_ms);

#ifdef __cplusplus
}
#endif
#endif /* KOMPASS_B200_H */
