// kc_dwa.cu — the DWA controller around the planner kernels (SURVEY §8 row f1): reference-path
// preparation (interpolate / segment), closest-point tracking, curvature-adaptive horizon, tracked
// segment selection, then one kc_planner cycle. Host scalar code; every launch goes through the
// planner (its C-ABI, or kc::planner_batch for a fleet) so this file adds no second path to the GPU.
// The follower state lives in `Follower`, which needs no planner: a kc_dwa handle keeps one, a
// kc_fleet keeps one per robot and steps them all in one batched launch set.
//
// ref: src/controllers/follower.cpp:15-304, src/controllers/dwa.cpp:14-233,
//      include/controllers/dwa.h:113-230, src/datatypes/path.cpp:55-400,
//      include/datatypes/path.h:190-226, include/utils/spline.h:211-224,390-419,
//      include/utils/angles.h:21-29.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <limits>
#include <vector>

#include "kc_common.cuh"

using namespace kc;

namespace {

// ---------------------------------------------------------------------------------------------
// Path::Path (ref: include/datatypes/path.h:112-297)
// ---------------------------------------------------------------------------------------------
struct RefPath {
  std::vector<float> X, Y, K;     // X_, Y_, Curvature_
  std::vector<float> acc;         // accumulated_path_length_ (may be shorter than X: path.cpp:300-306)
  std::vector<size_t> seg;        // segment_indices_
  float total_len = 0.0f;         // current_total_length_
  bool interpolated = false;

  size_t size() const { return X.size(); }

  static float dist(float ax, float ay, float bx, float by) {  // (p1 - p2).norm(), z = 0
    const float dx = ax - bx, dy = ay - by;
    return std::sqrt(dx * dx + (dy * dy + 0.0f));
  }

  // ref: path.cpp:150-165
  float totalPathLength() const {
    if (size() < 2) return 0.0f;
    if (interpolated) return total_len;
    float t = 0.0f;
    for (size_t i = 1; i < size(); ++i) t += dist(X[i - 1], Y[i - 1], X[i], Y[i]);
    return t;
  }

  // ref: path.cpp:167-288, linear tk::spline (spline.h:211-224: slope per knot interval, the
  // quadratic and cubic coefficients are zero; :402-419: value = ((d h + c) h + b) h + y)
  void interpolate_linear(double max_dist) {
    const size_t n = size();
    std::vector<double> s(n), xv(n), yv(n);
    s[0] = 0.0;
    xv[0] = X[0];
    yv[0] = Y[0];
    total_len = 0.0f;
    for (size_t i = 1; i < n; ++i) {
      const double seg_dist = std::hypot(X[i] - X[i - 1], Y[i] - Y[i - 1]);  // float overload
      total_len += seg_dist;                                                  // float += double
      s[i] = total_len;
      xv[i] = X[i];
      yv[i] = Y[i];
    }
    std::vector<double> bx(n), by(n);
    for (size_t i = 0; i + 1 < n; ++i) {
      bx[i] = (xv[i + 1] - xv[i]) / (s[i + 1] - s[i]);
      by[i] = (yv[i + 1] - yv[i]) / (s[i + 1] - s[i]);
    }
    bx[n - 1] = bx[n - 2];
    by[n - 1] = by[n - 2];
    auto value = [&](const std::vector<double> &b, const std::vector<double> &y, double x) {
      const size_t idx =
          (size_t)std::max((int)(std::upper_bound(s.begin(), s.end(), x) - s.begin()) - 1, 0);
      const double h = x - s[idx];
      const double zero = 0.0;  // m_c / m_d (and m_c0) of a linear spline
      if (x < s[0]) return (zero * h + b[0]) * h + y[0];
      if (x > s[n - 1]) return (zero * h + b[n - 1]) * h + y[n - 1];
      return ((zero * h + zero) * h + b[idx]) * h + y[idx];
    };
    const size_t new_size = (size_t)(total_len / max_dist) + 1;
    std::vector<float> nX(new_size, 0.0f), nY(new_size, 0.0f);
    acc.assign(new_size, 0.0f);
    size_t idx = 0;
    for (double t = 0.0; t <= total_len && idx < new_size; t += max_dist) {
      acc[idx] = (float)t;
      nX[idx] = (float)value(bx, xv, t);
      nY[idx] = (float)value(by, yv, t);
      idx++;
    }
    if (idx < new_size && idx > 0) {  // exact end point; its accumulated length stays 0 (reference quirk)
      nX[idx] = (float)value(bx, xv, total_len);
      nY[idx] = (float)value(by, yv, total_len);
      idx++;
    }
    interpolated = true;
    nX.resize(idx);
    nY.resize(idx);
    X.swap(nX);
    Y.swap(nY);
    K.assign(idx, 0.0f);
    if (idx >= 2) {  // ref: path.cpp:260-287
      float dx_old = X[1] - X[0], dy_old = Y[1] - Y[0];
      for (size_t i = 1; i + 1 < idx; ++i) {
        const float dx = X[i + 1] - X[i], dy = Y[i + 1] - Y[i];
        const float ddx = dx - dx_old, ddy = dy - dy_old;
        const float val = dx * dx + dy * dy;
        const float den = val * std::sqrt(val);
        K[i] = (den > 1e-6f) ? (dx_old * ddy - ddx * dy_old) / den : 0.0f;
        dx_old = dx;
        dy_old = dy;
      }
    }
  }

  // ref: path.cpp:290-330
  void segment(double seg_len, size_t max_pts) {
    const size_t n = size();
    if (n < 2) return;
    seg.clear();
    seg.push_back(0);
    if (!interpolated) {
      acc.resize(n - 1);
      for (size_t i = 0; i + 1 < n; ++i) acc[i] = dist(X[i], Y[i], X[i + 1], Y[i + 1]);
    }
    auto at = [&](size_t i) { return i < acc.size() ? acc[i] : 0.0f; };
    size_t start_idx = 0;
    float start_len = at(0);
    for (size_t i = 1; i < n; ++i) {
      const size_t pts = i - start_idx + 1;
      const float len = at(i) - start_len;
      if ((seg_len > 0.0 && len >= seg_len) || (max_pts > 0 && pts > max_pts)) {
        seg.push_back(i);
        start_idx = i;
        start_len = at(i);
      }
    }
  }

  size_t seg_start(size_t k) const { return seg[k]; }
  size_t seg_end(size_t k) const { return (k + 1 < seg.size()) ? seg[k + 1] - 1 : size() - 1; }
};

// Path::distanceSquared(State, Point): (Point(state.x, state.y, 0) - point).squaredNorm()
inline float dist2_state(double sx, double sy, float px, float py) {
  const float dx = (float)sx - px, dy = (float)sy - py;
  return dx * dx + (dy * dy + 0.0f);
}

inline double normalize_pm_pi(double a) {  // ref: angles.h:21-29
  a = std::fmod(a + M_PI, 2 * M_PI);
  if (a < 0) a += 2 * M_PI;
  a -= M_PI;
  return a;
}

struct PathPosition {  // ref: path.h:300-308
  size_t index = 0, segment_index = 0;
  double segment_length = -1.0, parallel_distance = 0.0, normal_distance = 0.0;
  double sx = 0.0, sy = 0.0, syaw = 0.0;
};

// Follower + Controller state of one robot (follower.h, controller.h) and what DWA adds to it
struct Follower {
  kc_follower_params fp;
  double time_step = 0.0;
  RefPath path;
  std::vector<float> acc_full;  // getDistanceAtIndex(i) for every path point
  bool has_path = false, path_processing = false, reached_goal = false;
  size_t max_segment_size = 0, max_segment_index = 0, current_segment_index = 0;
  double goal_distance = std::numeric_limits<double>::max();
  double state[4] = {0, 0, 0, 0};
  double vx_max_ctrl = 1.0, vy_max_ctrl = 1.0, omega_max_ctrl = 1.0;  // Controller::ctrlimitsParams
  double base_horizon = 0.0, max_forward_distance = 0.0;
  PathPosition closest;
  double latest_cmd[3] = {0, 0, 0};
  kc_dwa_info info;
};

}  // namespace

struct kc_dwa {
  kc_planner *planner = nullptr;
  kc_planner_config cfg;
  Follower f;
  // CostEvaluator::customTrajCostsPtrs_ (cost_evaluator.h:150-154): host callbacks, registration order
  struct Custom {
    double weight;
    kc_custom_cost_fn fn;
    void *user;
  };
  std::vector<Custom> customs;
  std::vector<double> custom_terms;  // [n_admissible x n_custom] weight * value of this cycle
  // DWA::debuggingSamples_ (dwa.h:232): a copy that outlives later calls on the planner
  bool has_debug = false;
  int32_t dbg_count = 0, dbg_points = 0;
  std::vector<float> dbg_vx, dbg_vy, dbg_om, dbg_x, dbg_y;
  std::vector<int32_t> dbg_slots;
};

namespace {

// ref: follower.cpp:149-176
size_t closest_segment(const Follower *d, size_t left, size_t right) {
  if (left == right) return left;
  const size_t mid = (left + right) / 2;
  const RefPath &p = d->path;
  const float dl = dist2_state(d->state[0], d->state[1], p.X[p.seg_start(left)], p.Y[p.seg_start(left)]);
  const float dr = dist2_state(d->state[0], d->state[1], p.X[p.seg_start(right)], p.Y[p.seg_start(right)]);
  if (mid == right || mid == left) return (dl <= dr) ? left : right;
  return (dl <= dr) ? closest_segment(d, left, mid) : closest_segment(d, mid, right);
}

// ref: follower.cpp:194-260
int32_t closest_on_segment(const Follower *d, size_t k, PathPosition &out) {
  const RefPath &p = d->path;
  KC_REQUIRE(k < p.seg.size(), KC_ERR_OUT_OF_RANGE,
             "Invalid segment index. Maximum number of segments is %zu, but requested segment index is %zu",
             p.seg.size() - 1, k);
  const size_t s = p.seg_start(k), e = p.seg_end(k), n = e - s + 1;
  double min_d2 = std::numeric_limits<float>::max();
  double cx = 0.0, cy = 0.0, seg_pos = 0.0;
  size_t best = 0;
  // Point components are floats: std::atan2(float, float) is the float overload (follower.cpp:214)
  const double heading = (double)std::atan2(p.Y[e] - p.Y[s], p.X[e] - p.X[s]);
  for (size_t i = 0; i < n; ++i) {
    const double d2 = dist2_state(d->state[0], d->state[1], p.X[s + i], p.Y[s + i]);
    if (d2 <= min_d2) {
      min_d2 = d2;
      cx = p.X[s + i];
      cy = p.Y[s + i];
      best = i;
      seg_pos = (n > 1) ? (double)i / (double)(n - 1) : 1.0;
    }
  }
  out.index = best + s;
  out.segment_index = k;
  out.segment_length = seg_pos;
  out.sx = cx;
  out.sy = cy;
  out.syaw = heading;
  out.normal_distance = std::sqrt(min_d2);
  const double vx = d->state[0] - cx, vy = d->state[1] - cy;
  const double cross = std::cos(heading) * vy - std::sin(heading) * vx;
  out.parallel_distance = cross > 0 ? out.normal_distance : -out.normal_distance;
  return KC_OK;
}

// ref: follower.cpp:262-304
int32_t determine_target(Follower *d) {
  const RefPath &p = d->path;
  PathPosition &c = d->closest;
  KC_REQUIRE(d->current_segment_index < p.seg.size(), KC_ERR_OUT_OF_RANGE,
             "Invalid segment index. Maximum number of segments is %zu, but requested segment index is %zu",
             p.seg.size() - 1, d->current_segment_index);
  if (c.segment_length <= 0.0 || c.index >= p.seg_end(d->current_segment_index) ||
      c.segment_length >= 0.9) {
    d->current_segment_index = closest_segment(d, 0, d->max_segment_index);
    KC_TRY(closest_on_segment(d, d->current_segment_index, c));
  } else {
    KC_TRY(closest_on_segment(d, c.segment_index, c));
  }
  d->info.closest_index = (int32_t)c.index;
  d->info.segment_index = (int32_t)d->current_segment_index;
  d->info.segment_position = c.segment_length;
  d->info.crosstrack_error = c.parallel_distance;
  d->info.heading_error = normalize_pm_pi(c.syaw - d->state[2]);
  d->info.target_x = c.sx;
  d->info.target_y = c.sy;
  d->info.target_yaw = c.syaw;
  return KC_OK;
}

// ref: dwa.cpp:157-206: the horizon of this cycle, and the points per trajectory it gives (the
// sampler's clamp and truncation, kc::horizon_points, as kc_planner_set_prediction_horizon applies it)
int32_t adapt_horizon(Follower *d) {
  const double base = d->base_horizon, v_max = d->vx_max_ctrl;
  const double interp = d->fp.max_point_interpolation_distance;
  const RefPath &p = d->path;
  double horizon = base;
  if (d->has_path && !(v_max < 1e-3) && !(interp <= 0.0)) {
    const size_t start = std::min(d->closest.index, p.size() - 1);
    const size_t peek = (size_t)std::ceil(base * v_max / interp);
    const size_t end = std::min(start + peek, p.size() - 1);
    float kappa = 0.0f;
    for (size_t i = start; i <= end; ++i) kappa = std::max(kappa, std::abs((float)(double)p.K[i]));
    if (kappa > d->fp.curvature_horizon_tolerance)
      horizon = std::min(base, std::sqrt(8.0 * d->fp.curvature_horizon_tolerance / kappa) / v_max);
  }
  double clamped = horizon;
  const int32_t P = kc::horizon_points(d->time_step, d->base_horizon, clamped);
  d->max_forward_distance = horizon * v_max;
  d->info.horizon = horizon;
  d->info.n_points = P;
  return P;
}

// ref: dwa.cpp:208-233
void tracked_segment(Follower *d) {
  const RefPath &p = d->path;
  size_t s = d->closest.index;
  if (s >= p.size()) s = p.size() - 1;
  size_t look = d->max_segment_size;
  const double interp = d->fp.max_point_interpolation_distance;
  if (interp > 0.0) look = std::max(look, (size_t)std::ceil(d->max_forward_distance / interp) + 1);
  const size_t e = std::min(s + look, p.size() - 1);
  d->info.seg_start = (int32_t)s;
  d->info.seg_count = (int32_t)(e - s + 1);
}

// determineTarget + the adaptive horizon + the tracked segment: everything of a DWA cycle before
// the planner runs (the rotate-in-place shortcut of dwa.h:195-206 is dead code in the reference:
// Follower::setParams derives rotate_in_place from Controller::ctrType, which DWA never sets)
int32_t follower_prepare(Follower *d) {
  KC_TRY(determine_target(d));
  adapt_horizon(d);
  tracked_segment(d);
  return KC_OK;
}

// ref: dwa.h:134-137 latest_velocity_command_ (kept when no trajectory is found)
void follower_take_command(Follower *d, const kc_cycle_result &out) {
  if (out.found && out.n_points >= 2) {
    d->latest_cmd[0] = out.vx[0];
    d->latest_cmd[1] = out.vy[0];
    d->latest_cmd[2] = out.omega[0];
  }
}

// ref: follower.h:147-165 get*Cmd (clamped to the base-class limits)
void follower_command(const Follower *d, double cmd[3]) {
  cmd[0] = std::max(std::min(d->latest_cmd[0], d->vx_max_ctrl), -d->vx_max_ctrl);
  cmd[1] = std::max(std::min(d->latest_cmd[1], d->vy_max_ctrl), -d->vy_max_ctrl);
  cmd[2] = std::max(std::min(d->latest_cmd[2], d->omega_max_ctrl), -d->omega_max_ctrl);
}

// parameter ranges of FollowerParameters (follower.h:24-75) and the follower's start state
int32_t follower_init(Follower *d, const kc_planner_config &cfg, const kc_follower_params *fp) {
  kc_follower_params f;
  kc_follower_params_default(&f);
  if (fp) f = *fp;
  KC_REQUIRE(f.max_point_interpolation_distance >= 0.0001 && f.max_point_interpolation_distance <= 1000.0,
             KC_ERR_OUT_OF_RANGE, "max_point_interpolation_distance out of range [0.0001, 1000]");
  KC_REQUIRE(f.path_segment_length >= 0.001 && f.path_segment_length <= 1000.0, KC_ERR_OUT_OF_RANGE,
             "path_segment_length out of range [0.001, 1000]");
  KC_REQUIRE(f.goal_dist_tolerance >= 0.001 && f.goal_dist_tolerance <= 1000.0, KC_ERR_OUT_OF_RANGE,
             "goal_dist_tolerance out of range [0.001, 1000]");
  KC_REQUIRE(f.loosing_goal_distance >= 0.001 && f.loosing_goal_distance <= 1000.0, KC_ERR_OUT_OF_RANGE,
             "loosing_goal_distance out of range [0.001, 1000]");
  KC_REQUIRE(f.curvature_horizon_tolerance >= 0.5 && f.curvature_horizon_tolerance <= 1000.0,
             KC_ERR_OUT_OF_RANGE, "curvature_horizon_tolerance out of range [0.5, 1000]");
  d->fp = f;
  d->time_step = cfg.time_step;
  d->base_horizon = cfg.prediction_horizon;
  // ref: follower.cpp:54-59 (double quotient + 1, truncated to size_t)
  d->max_segment_size = (size_t)(f.path_segment_length / f.max_point_interpolation_distance + 1);
  // ref: dwa.cpp:31-37
  d->max_forward_distance =
      (cfg.control_type == KC_OMNI ? std::max(cfg.vx_max, cfg.vy_max) : cfg.vx_max) * cfg.prediction_horizon;
  memset(&d->info, 0, sizeof(d->info));
  return KC_OK;
}

// ref: follower.cpp:81-107 setCurrentPath, first half: the interpolated and segmented path and its
// getDistanceAtIndex(i) for every point (0 beyond the stored lengths); nothing of `d` changes
int32_t follower_build_path(const Follower *d, const float *x, const float *y, int32_t n, int32_t interpolate,
                            RefPath &p, std::vector<float> &acc) {
  KC_REQUIRE(x && y, KC_ERR_INVALID_ARG, "null argument");
  KC_REQUIRE(n >= 2, KC_ERR_INVALID_ARG, "At least two points are required to create a path.");
  p.X.assign(x, x + n);
  p.Y.assign(y, y + n);
  p.K.assign(n, 0.0f);
  if (interpolate) p.interpolate_linear(d->fp.max_point_interpolation_distance);
  KC_REQUIRE(p.size() >= 2, KC_ERR_INVALID_ARG,
             "reference path collapses to fewer than two points after interpolation");
  p.segment(d->fp.path_segment_length, d->max_segment_size);
  acc.assign(p.size(), 0.0f);
  for (size_t i = 0; i < p.size() && i < p.acc.size(); ++i) acc[i] = p.acc[i];
  return KC_OK;
}

// second half: the follower takes the new path
void follower_set_path(Follower *d, RefPath &&p, std::vector<float> &&acc) {
  d->path = std::move(p);
  d->acc_full = std::move(acc);
  d->has_path = true;
  d->max_segment_index = d->path.seg.size() - 1;
  d->path_processing = true;
  d->current_segment_index = 0;
  d->goal_distance = std::numeric_limits<double>::max();
  d->reached_goal = false;
}

// ref: follower.cpp:68-79
void follower_clear_path(Follower *d) {
  d->has_path = false;
  d->reached_goal = true;
  d->path_processing = false;
}

// ref: follower.cpp:111-145
int32_t follower_goal_reached(Follower *d) {
  if (!d->path_processing) return 1;
  const RefPath &p = d->path;
  const size_t last = p.size() - 1;
  bool loosing = false;
  const double dist = std::hypot(d->state[0] - (double)p.X[last], d->state[1] - (double)p.Y[last]);
  const bool end_reached = dist <= d->fp.goal_dist_tolerance;
  if ((d->current_segment_index + 1) >= d->max_segment_index) {
    if (dist < d->goal_distance) {
      d->goal_distance = dist;
    } else if (std::abs(dist - d->goal_distance) > d->fp.loosing_goal_distance) {
      loosing = true;
    }
  }
  if (end_reached || loosing) {
    d->path_processing = false;
    d->reached_goal = true;
  }
  return d->reached_goal ? 1 : 0;
}

int32_t generate(kc_dwa *d, const double vel[3], const double pose[3], bool cloud, const void *a,
                 const void *b, int32_t n, kc_samples *s) {
  if (cloud) return kc_sampler_generate_cloud(d->planner, vel, pose, (const float *)a, n, s);
  return kc_sampler_generate_scan(d->planner, vel, pose, (const double *)a, (const double *)b, n, s);
}

// DWA::findBestPath with registered custom costs (dwa.h:214-229 + cost_evaluator.cpp:96-100): the
// callbacks are host functions of the sampled trajectories, so this cycle runs the reference's own
// three steps instead of the fused launch set: generateTrajectories (admissible rows come back to
// the host) -> callbacks -> setPointScan + getMinTrajectoryCost with the callback terms uploaded
// beside the rows (what the reference's GPU evaluator does too, cost_evaluator_gpu.cpp:344-370).
int32_t cycle_with_custom_costs(kc_dwa *d, const double vel[3], const double pose[3], bool cloud,
                                const void *a, const void *b, int32_t n, int32_t seg_start,
                                int32_t seg_count, kc_cycle_result *out) {
  kc_samples s;
  KC_TRY(generate(d, vel, pose, cloud, a, b, n, &s));
  const int32_t n_slots = kc_planner_num_slots_last(d->planner);
  if (s.count == 0) {  // dwa.h:219-221: TrajSearchResult{Trajectory2D(), false, 0.0}
    memset(out, 0, sizeof(*out));
    out->slot = -1;
    out->n_points = s.n_points;
    out->n_slots = n_slots;
    return KC_OK;
  }
  const float range = kc_planner_get_max_range(d->planner);
  if (cloud)
    KC_TRY(kc_cost_set_points_cloud(d->planner, (const float *)a, n, pose, range, 3.0f));
  else
    KC_TRY(kc_cost_set_points_scan(d->planner, (const double *)a, (const double *)b, n, pose, range, 3.0f));
  const size_t nc = d->customs.size(), P = (size_t)s.n_points;
  d->custom_terms.resize((size_t)s.count * nc);
  kc_path_view pv;
  pv.n = (int32_t)d->f.path.size();
  pv.X = d->f.path.X.data();
  pv.Y = d->f.path.Y.data();
  pv.acc = d->f.acc_full.data();
  pv.total_length = d->f.path.totalPathLength();
  for (int32_t t = 0; t < s.count; ++t) {
    kc_trajectory_view tv;
    tv.n_points = s.n_points;
    tv.vx = s.vx + (size_t)t * (P - 1);
    tv.vy = s.vy + (size_t)t * (P - 1);
    tv.omega = s.omega + (size_t)t * (P - 1);
    tv.x = s.x + (size_t)t * P;
    tv.y = s.y + (size_t)t * P;
    for (size_t k = 0; k < nc; ++k)
      d->custom_terms[(size_t)t * nc + k] = d->customs[k].weight * d->customs[k].fn(&tv, &pv, d->customs[k].user);
  }
  KC_TRY(kc_cost_evaluate(d->planner, s.count, s.n_points, s.vx, s.vy, s.omega, s.x, s.y, seg_start,
                          seg_count, d->custom_terms.data(), (int32_t)nc, nullptr, out));
  if (out->found) out->slot = s.slots[out->slot];  // row of the admissible list -> enumeration slot
  out->n_slots = n_slots;
  out->n_admissible = s.count;
  return KC_OK;
}

int32_t compute(kc_dwa *d, const double vel[3], bool cloud, const void *a, const void *b, int32_t n,
                kc_cycle_result *out, kc_dwa_info *info) {
  KC_REQUIRE(d && vel && out, KC_ERR_INVALID_ARG, "null argument");
  Follower &f = d->f;
  KC_REQUIRE(f.has_path, KC_ERR_INVALID_ARG,
             "Pointer to global path is NULL. Cannot use DWA local planner without setting a global path");
  KC_TRY(follower_prepare(&f));
  KC_TRY(kc_planner_set_prediction_horizon(d->planner, f.info.horizon, nullptr));
  const int32_t seg_start = f.info.seg_start, seg_count = f.info.seg_count;
  const double pose[3] = {f.state[0], f.state[1], f.state[2]};
  if (!d->customs.empty()) {
    KC_TRY(cycle_with_custom_costs(d, vel, pose, cloud, a, b, n, seg_start, seg_count, out));
  } else if (cloud)
    KC_TRY(kc_planner_cycle_cloud(d->planner, vel, pose, (const float *)a, n, seg_start, seg_count, out));
  else
    KC_TRY(kc_planner_cycle_scan(d->planner, vel, pose, (const double *)a, (const double *)b, n,
                                 seg_start, seg_count, out));
  follower_take_command(&f, *out);
  if (info) *info = f.info;
  return KC_OK;
}

}  // namespace

extern "C" {

void kc_follower_params_default(kc_follower_params *p) {
  if (!p) return;
  // ref: follower.h:24-75 FollowerParameters defaults
  p->max_point_interpolation_distance = 0.01;
  p->lookahead_distance = 1.0;
  p->goal_dist_tolerance = 0.1;
  p->path_segment_length = 1.0;
  p->goal_orientation_tolerance = 0.1;
  p->loosing_goal_distance = 0.5;
  p->curvature_horizon_tolerance = 1.5;
}

// Path::interpolate(LINEAR) + Path::segment on the host (no device needed): fills caller arrays.
int32_t kc_path_prepare(const float *x, const float *y, int32_t n, int32_t interpolate,
                        double max_point_interpolation_distance, double path_segment_length,
                        int64_t max_points_per_segment, int32_t cap, float *X, float *Y, float *acc,
                        float *curvature, int32_t *seg_starts, int32_t *n_out, int32_t *n_segments,
                        float *total_length) {
  KC_REQUIRE(x && y && X && Y && acc && curvature && seg_starts && n_out && n_segments && total_length,
             KC_ERR_INVALID_ARG, "null argument");
  KC_REQUIRE(n >= 2, KC_ERR_INVALID_ARG, "At least two points are required to create a path.");
  KC_REQUIRE(max_point_interpolation_distance > 0.0, KC_ERR_OUT_OF_RANGE,
             "max_point_interpolation_distance must be positive");
  RefPath p;
  p.X.assign(x, x + n);
  p.Y.assign(y, y + n);
  p.K.assign(n, 0.0f);
  if (interpolate) p.interpolate_linear(max_point_interpolation_distance);
  p.segment(path_segment_length, (size_t)std::max<int64_t>(max_points_per_segment, 0));
  KC_REQUIRE((int64_t)p.size() <= cap && (int64_t)p.seg.size() <= cap, KC_ERR_OUT_OF_RANGE,
             "output capacity %d too small for %zu points", cap, p.size());
  for (size_t i = 0; i < p.size(); ++i) {
    X[i] = p.X[i];
    Y[i] = p.Y[i];
    curvature[i] = p.K[i];
    acc[i] = i < p.acc.size() ? p.acc[i] : 0.0f;
  }
  for (size_t k = 0; k < p.seg.size(); ++k) seg_starts[k] = (int32_t)p.seg[k];
  *n_out = (int32_t)p.size();
  *n_segments = (int32_t)p.seg.size();
  *total_length = p.totalPathLength();
  return KC_OK;
}

int32_t kc_dwa_create(const kc_planner_config *cfg, const kc_follower_params *fp, kc_dwa **out) {
  KC_REQUIRE(out, KC_ERR_INVALID_ARG, "null output handle");
  *out = nullptr;
  KC_REQUIRE(cfg, KC_ERR_INVALID_ARG, "null config");
  Follower f;
  KC_TRY(follower_init(&f, *cfg, fp));
  kc_planner *pl = nullptr;
  KC_TRY(kc_planner_create(cfg, &pl));
  kc_dwa *d = new kc_dwa();
  d->planner = pl;
  d->cfg = *cfg;
  d->f = std::move(f);
  *out = d;
  return KC_OK;
}

void kc_dwa_destroy(kc_dwa *d) {
  kc::ensure_device();  // the handle's device on this thread (frees below)
  if (!d) return;
  kc_planner_destroy(d->planner);
  delete d;
}

kc_planner *kc_dwa_planner(kc_dwa *d) { return d ? d->planner : nullptr; }

// ref: follower.cpp:81-107 setCurrentPath
int32_t kc_dwa_set_current_path(kc_dwa *d, const float *x, const float *y, int32_t n, int32_t interpolate) {
  KC_REQUIRE(d && x && y, KC_ERR_INVALID_ARG, "null argument");
  KC_REQUIRE(n >= 2, KC_ERR_INVALID_ARG, "At least two points are required to create a path.");
  KC_TRY(kc::ensure_device());
  RefPath p;
  std::vector<float> acc;
  KC_TRY(follower_build_path(&d->f, x, y, n, interpolate, p, acc));
  KC_TRY(kc_planner_set_path(d->planner, p.X.data(), p.Y.data(), acc.data(), (int32_t)p.size(),
                             p.totalPathLength()));
  follower_set_path(&d->f, std::move(p), std::move(acc));
  return KC_OK;
}

// ref: follower.cpp:68-79
int32_t kc_dwa_clear_current_path(kc_dwa *d) {
  KC_REQUIRE(d, KC_ERR_INVALID_ARG, "null handle");
  KC_TRY(kc::ensure_device());
  follower_clear_path(&d->f);
  return KC_OK;
}

int32_t kc_dwa_set_current_state(kc_dwa *d, double x, double y, double yaw, double speed) {
  KC_REQUIRE(d, KC_ERR_INVALID_ARG, "null handle");
  KC_TRY(kc::ensure_device());
  d->f.state[0] = x;
  d->f.state[1] = y;
  d->f.state[2] = yaw;
  d->f.state[3] = speed;
  return KC_OK;
}

// ref: controller.cpp:22-33 setLinearControlLimits / setAngularControlLimits (base-class limits:
// used by the horizon adaptation and the command getters only; DWA itself never sets them)
int32_t kc_dwa_set_control_limits(kc_dwa *d, double vx_max, double vy_max, double omega_max) {
  KC_REQUIRE(d, KC_ERR_INVALID_ARG, "null handle");
  KC_TRY(kc::ensure_device());
  d->f.vx_max_ctrl = vx_max;
  d->f.vy_max_ctrl = vy_max;
  d->f.omega_max_ctrl = omega_max;
  return KC_OK;
}

// ref: follower.cpp:111-145
int32_t kc_dwa_is_goal_reached(kc_dwa *d, int32_t *reached) {
  KC_REQUIRE(d && reached, KC_ERR_INVALID_ARG, "null argument");
  KC_TRY(kc::ensure_device());
  *reached = follower_goal_reached(&d->f);
  return KC_OK;
}

int32_t kc_dwa_has_path(const kc_dwa *d) {  // ref: follower.h:177-182
  if (!d || !d->f.has_path || !d->f.path_processing) return 0;
  return d->f.path.totalPathLength() > 0.0f ? 1 : 0;
}

int32_t kc_dwa_get_path(const kc_dwa *d, const float **X, const float **Y, const float **curvature,
                        int32_t *n, int32_t *n_segments, float *total_length) {
  KC_REQUIRE(d, KC_ERR_INVALID_ARG, "null handle");
  const Follower &f = d->f;
  KC_REQUIRE(f.has_path, KC_ERR_INVALID_ARG, "no current path");
  if (X) *X = f.path.X.data();
  if (Y) *Y = f.path.Y.data();
  if (curvature) *curvature = f.path.K.data();
  if (n) *n = (int32_t)f.path.size();
  if (n_segments) *n_segments = (int32_t)f.path.seg.size();
  if (total_length) *total_length = f.path.totalPathLength();
  return KC_OK;
}

// ref: follower.h:147-165 get*Cmd (clamped to the base-class limits)
int32_t kc_dwa_get_command(const kc_dwa *d, double cmd[3]) {
  KC_REQUIRE(d && cmd, KC_ERR_INVALID_ARG, "null argument");
  follower_command(&d->f, cmd);
  return KC_OK;
}

// ref: dwa.cpp:147-150 addCustomCost
int32_t kc_dwa_add_custom_cost(kc_dwa *d, double weight, kc_custom_cost_fn fn, void *user) {
  KC_REQUIRE(d && fn, KC_ERR_INVALID_ARG, "null argument");
  d->customs.push_back({weight, fn, user});
  return KC_OK;
}

int32_t kc_dwa_clear_custom_costs(kc_dwa *d) {
  KC_REQUIRE(d, KC_ERR_INVALID_ARG, "null handle");
  d->customs.clear();
  return KC_OK;
}

namespace {
// ref: dwa.h:147-165 debugVelocitySearch<T>: determineTarget, then the sampler alone with the given
// dropping mode (which stays set afterwards, as in the reference); the horizon is left as it is.
int32_t debug_search(kc_dwa *d, const double vel[3], bool cloud, const void *a, const void *b, int32_t n,
                     int32_t drop_samples, kc_samples *out) {
  KC_REQUIRE(d && vel, KC_ERR_INVALID_ARG, "null argument");
  KC_REQUIRE(d->f.has_path, KC_ERR_INVALID_ARG,
             "Pointer to global path is NULL. Cannot use DWA local planner without setting a global path");
  KC_TRY(determine_target(&d->f));
  KC_TRY(kc_planner_set_drop_samples(d->planner, drop_samples));
  const double pose[3] = {d->f.state[0], d->f.state[1], d->f.state[2]};
  kc_samples s;
  KC_TRY(generate(d, vel, pose, cloud, a, b, n, &s));
  const size_t P = (size_t)s.n_points, nv = (size_t)s.count * (P - 1), np = (size_t)s.count * P;
  d->dbg_count = s.count;
  d->dbg_points = s.n_points;
  d->dbg_vx.assign(s.vx, s.vx + nv);
  d->dbg_vy.assign(s.vy, s.vy + nv);
  d->dbg_om.assign(s.omega, s.omega + nv);
  d->dbg_x.assign(s.x, s.x + np);
  d->dbg_y.assign(s.y, s.y + np);
  d->dbg_slots.assign(s.slots, s.slots + s.count);
  d->has_debug = true;
  if (out) return kc_dwa_get_debugging_samples(d, out);
  return KC_OK;
}
}  // namespace

int32_t kc_dwa_debug_velocity_search_scan(kc_dwa *d, const double vel[3], const double *ranges,
                                          const double *angles, int32_t n, int32_t drop_samples,
                                          kc_samples *out) {
  KC_REQUIRE(n == 0 || (ranges && angles), KC_ERR_INVALID_ARG, "null scan arrays");
  KC_TRY(kc::ensure_device());
  return debug_search(d, vel, false, ranges, angles, n, drop_samples, out);
}

int32_t kc_dwa_debug_velocity_search_cloud(kc_dwa *d, const double vel[3], const float *xyz, int32_t n,
                                           int32_t drop_samples, kc_samples *out) {
  KC_REQUIRE(n == 0 || xyz, KC_ERR_INVALID_ARG, "null cloud");
  KC_TRY(kc::ensure_device());
  return debug_search(d, vel, true, xyz, nullptr, n, drop_samples, out);
}

// ref: dwa.cpp:235-250 getDebuggingSamples / getDebuggingSamplesPure
int32_t kc_dwa_get_debugging_samples(const kc_dwa *d, kc_samples *out) {
  KC_REQUIRE(d && out, KC_ERR_INVALID_ARG, "null argument");
  KC_REQUIRE(d->has_debug, KC_ERR_INVALID_ARG, "No debugging samples are available");
  out->count = d->dbg_count;
  out->n_points = d->dbg_points;
  out->vx = d->dbg_vx.data();
  out->vy = d->dbg_vy.data();
  out->omega = d->dbg_om.data();
  out->x = d->dbg_x.data();
  out->y = d->dbg_y.data();
  out->slots = d->dbg_slots.data();
  return KC_OK;
}

int32_t kc_dwa_compute_scan(kc_dwa *d, const double vel[3], const double *ranges, const double *angles,
                            int32_t n, kc_cycle_result *out, kc_dwa_info *info) {
  KC_REQUIRE(n == 0 || (ranges && angles), KC_ERR_INVALID_ARG, "null scan arrays");
  KC_TRY(kc::ensure_device());
  return compute(d, vel, false, ranges, angles, n, out, info);
}

int32_t kc_dwa_compute_cloud(kc_dwa *d, const double vel[3], const float *xyz, int32_t n,
                             kc_cycle_result *out, kc_dwa_info *info) {
  KC_REQUIRE(n == 0 || xyz, KC_ERR_INVALID_ARG, "null cloud");
  KC_TRY(kc::ensure_device());
  return compute(d, vel, true, xyz, nullptr, n, out, info);
}

}  // extern "C"

// =================================================================================================
// Fleet: R robots, each with its own path, state, horizon and sensor data, stepped together. Every
// robot's step is the kc_dwa cycle above (same follower code, same kernels), but one batched launch
// set per chunk of robots replaces R latency-bound cycles.
// =================================================================================================
struct kc_fleet {
  kc_planner *planner = nullptr;
  kc_planner_config cfg;
  int32_t R = 0;
  std::vector<Follower> robots;
  // path table: every robot's interpolated X | Y | acc on the device, uploaded when its path changes
  std::vector<DevBuf<float>> d_path;
  std::vector<float> path_len;  // Path::totalPathLength() of each robot's path
  // the last step: per-robot descriptors and winner records (rows in the planner's host copy)
  std::vector<kc::BatchRobot> batch;
  std::vector<double> poses;
  std::vector<kc_batch_result> heads;
  std::vector<kc_cycle_result> last;
  bool stepped = false;
};

namespace {

int32_t fleet_compute(kc_fleet *f, const double *vel, const kc::BatchSensor &sen, const int64_t *offsets,
                      const int32_t *counts, kc_fleet_result *results, kc_dwa_info *info) {
  KC_REQUIRE(f && vel && offsets && counts && results, KC_ERR_INVALID_ARG, "null argument");
  const int R = f->R;
  for (int r = 0; r < R; ++r) {
    KC_REQUIRE(counts[r] >= 0 && offsets[r] >= 0, KC_ERR_INVALID_ARG,
               "robot %d: bad sensor extents (offset %lld, count %d)", r, (long long)offsets[r], counts[r]);
    KC_REQUIRE(f->robots[r].has_path, KC_ERR_INVALID_ARG,
               "robot %d: Pointer to global path is NULL. Cannot use DWA local planner without setting a "
               "global path", r);
  }
  KC_TRY(kc::ensure_device());
  f->stepped = false;
  for (int r = 0; r < R; ++r) {
    Follower &fo = f->robots[r];
    KC_TRY(follower_prepare(&fo));
    double *pose = f->poses.data() + 3 * (size_t)r;
    pose[0] = fo.state[0];
    pose[1] = fo.state[1];
    pose[2] = fo.state[2];
    kc::BatchRobot &b = f->batch[r];
    b.vel = vel + 3 * (size_t)r;
    b.pose = pose;
    b.P = fo.info.n_points;
    b.path.hX = fo.path.X.data();
    b.path.hY = fo.path.Y.data();
    b.path.n = (int32_t)fo.path.size();
    b.path.dX = f->d_path[r].ptr;
    b.path.dY = b.path.dX + b.path.n;
    b.path.dAcc = b.path.dX + 2 * (size_t)b.path.n;
    b.path.total_length = f->path_len[r];
    b.seg_start = fo.info.seg_start;
    b.seg_count = fo.info.seg_count;
    b.offset = offsets[r];
    b.count = counts[r];
  }
  KC_TRY(kc::planner_batch(f->planner, R, f->batch.data(), sen, f->heads.data(), f->last.data()));
  f->stepped = true;
  for (int r = 0; r < R; ++r) {
    Follower &fo = f->robots[r];
    const kc_cycle_result &c = f->last[r];
    follower_take_command(&fo, c);
    kc_fleet_result &o = results[r];
    o.found = c.found;
    o.cost = c.cost;
    o.slot = c.slot;
    o.n_points = c.n_points;
    o.n_slots = c.n_slots;
    o.n_admissible = c.n_admissible;
    follower_command(&fo, o.cmd);
    if (info) info[r] = fo.info;
  }
  return KC_OK;
}

}  // namespace

extern "C" {

int32_t kc_fleet_create(const kc_planner_config *cfg, const kc_follower_params *fp, int32_t n_robots,
                        kc_fleet **out) {
  KC_REQUIRE(out, KC_ERR_INVALID_ARG, "null output handle");
  *out = nullptr;
  KC_REQUIRE(cfg, KC_ERR_INVALID_ARG, "null config");
  KC_REQUIRE(n_robots > 0, KC_ERR_INVALID_ARG, "n_robots must be positive (got %d)", n_robots);
  Follower proto;
  KC_TRY(follower_init(&proto, *cfg, fp));
  kc_planner *pl = nullptr;
  KC_TRY(kc_planner_create(cfg, &pl));
  kc_fleet *f = new kc_fleet();
  f->planner = pl;
  f->cfg = *cfg;
  f->R = n_robots;
  f->robots.assign(n_robots, proto);
  f->d_path.resize(n_robots);
  f->path_len.assign(n_robots, 0.0f);
  f->batch.resize(n_robots);
  f->poses.assign(3 * (size_t)n_robots, 0.0);
  f->heads.resize(n_robots);
  f->last.resize(n_robots);
  *out = f;
  return KC_OK;
}

void kc_fleet_destroy(kc_fleet *f) {
  kc::ensure_device();  // the handle's device on this thread (frees below)
  if (!f) return;
  kc_planner_destroy(f->planner);
  for (DevBuf<float> &b : f->d_path) b.release();
  delete f;
}

kc_planner *kc_fleet_planner(kc_fleet *f) { return f ? f->planner : nullptr; }

int32_t kc_fleet_set_current_path(kc_fleet *f, int32_t robot, const float *x, const float *y, int32_t n,
                                  int32_t interpolate) {
  KC_REQUIRE(f && x && y, KC_ERR_INVALID_ARG, "null argument");
  KC_REQUIRE(robot >= 0 && robot < f->R, KC_ERR_INVALID_ARG, "robot %d out of range [0, %d)", robot, f->R);
  KC_REQUIRE(n >= 2, KC_ERR_INVALID_ARG, "At least two points are required to create a path.");
  KC_TRY(kc::ensure_device());
  RefPath p;
  std::vector<float> acc;
  KC_TRY(follower_build_path(&f->robots[robot], x, y, n, interpolate, p, acc));
  const size_t m = p.size();
  DevBuf<float> &d = f->d_path[robot];
  KC_TRY(d.reserve(3 * m));  // a step has finished (synchronised) before this call: nothing reads d
  KC_CUDA(cudaMemcpy(d.ptr, p.X.data(), m * 4, cudaMemcpyHostToDevice));
  KC_CUDA(cudaMemcpy(d.ptr + m, p.Y.data(), m * 4, cudaMemcpyHostToDevice));
  KC_CUDA(cudaMemcpy(d.ptr + 2 * m, acc.data(), m * 4, cudaMemcpyHostToDevice));
  f->path_len[robot] = p.totalPathLength();
  follower_set_path(&f->robots[robot], std::move(p), std::move(acc));
  return KC_OK;
}

int32_t kc_fleet_clear_current_path(kc_fleet *f, int32_t robot) {
  KC_REQUIRE(f, KC_ERR_INVALID_ARG, "null handle");
  KC_REQUIRE(robot >= 0 && robot < f->R, KC_ERR_INVALID_ARG, "robot %d out of range [0, %d)", robot, f->R);
  follower_clear_path(&f->robots[robot]);
  return KC_OK;
}

int32_t kc_fleet_set_current_states(kc_fleet *f, const double *states) {
  KC_REQUIRE(f && states, KC_ERR_INVALID_ARG, "null argument");
  for (int r = 0; r < f->R; ++r)
    for (int k = 0; k < 4; ++k) f->robots[r].state[k] = states[4 * (size_t)r + k];
  return KC_OK;
}

int32_t kc_fleet_set_control_limits(kc_fleet *f, double vx_max, double vy_max, double omega_max) {
  KC_REQUIRE(f, KC_ERR_INVALID_ARG, "null handle");
  for (Follower &fo : f->robots) {
    fo.vx_max_ctrl = vx_max;
    fo.vy_max_ctrl = vy_max;
    fo.omega_max_ctrl = omega_max;
  }
  return KC_OK;
}

int32_t kc_fleet_compute_cloud(kc_fleet *f, const double *vel, const float *xyz, const int64_t *offsets,
                               const int32_t *counts, kc_fleet_result *results, kc_dwa_info *info) {
  kc::BatchSensor sen;
  sen.cloud = true;
  sen.xyz = xyz;
  return fleet_compute(f, vel, sen, offsets, counts, results, info);
}

int32_t kc_fleet_compute_scan(kc_fleet *f, const double *vel, const double *ranges, const double *angles,
                              const int64_t *offsets, const int32_t *counts, kc_fleet_result *results,
                              kc_dwa_info *info) {
  kc::BatchSensor sen;
  sen.cloud = false;
  sen.ranges = ranges;
  sen.angles = angles;
  return fleet_compute(f, vel, sen, offsets, counts, results, info);
}

int32_t kc_fleet_get_trajectory(const kc_fleet *f, int32_t robot, kc_cycle_result *out) {
  KC_REQUIRE(f && out, KC_ERR_INVALID_ARG, "null argument");
  KC_REQUIRE(robot >= 0 && robot < f->R, KC_ERR_INVALID_ARG, "robot %d out of range [0, %d)", robot, f->R);
  KC_REQUIRE(f->stepped, KC_ERR_INVALID_ARG, "no fleet step has completed yet");
  *out = f->last[robot];
  return KC_OK;
}

int32_t kc_fleet_is_goal_reached(kc_fleet *f, int32_t *reached) {
  KC_REQUIRE(f && reached, KC_ERR_INVALID_ARG, "null argument");
  for (int r = 0; r < f->R; ++r) reached[r] = follower_goal_reached(&f->robots[r]);
  return KC_OK;
}

}  // extern "C"
