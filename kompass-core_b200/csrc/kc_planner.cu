// kc_planner.cu — host side of the DWA planner C-ABI: per-cycle scalar prep (velocity window,
// transforms, windows), packed single H2D, kernel launches, result fetch.
//
// ref: include/controllers/dwa.h:183-230 (findBestPath flow), src/utils/trajectory_sampler.cpp,
//      include/utils/cost_evaluator.h:174-223, src/utils/cost_evaluator.cpp:49-109.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstring>
#include <thread>
#include <vector>

#include "kc_host_math.h"
#include "kc_hostcopy.h"
#include "kc_planner_kernels.cuh"

using namespace kc;

namespace {

constexpr size_t kAlign = 256;
inline int host_float_to_ordered(float f) {
  int i;
  memcpy(&i, &f, sizeof(i));
  return (i >= 0) ? i : i ^ 0x7fffffff;
}
inline size_t align_up(size_t v) { return (v + kAlign - 1) / kAlign * kAlign; }

struct Axes {
  std::vector<double> vx, vy, om;
  std::vector<int32_t> row_off;
  int32_t nvy = 0, nom = 0, n_slots = 0;
  double max_speed = 0.0;
};

// ref: include/datatypes/trajectory.h:19-29
void linear_split(int ctrl, int max_lin, int &nx, int &ny) {
  auto odd = [](int n) { return (n % 2 == 0) ? n + 1 : n; };
  if (ctrl == KC_OMNI) {
    nx = odd(std::max(3, max_lin * 3 / 4));
    ny = odd(std::max(3, max_lin * 1 / 4));
  } else {
    nx = odd(std::max(3, max_lin));
    ny = 1;
  }
}

// Velocity axes of this cycle, accumulated exactly like the reference loops
// (`for (v = min; v <= max; v += res)` in double; ref trajectory_sampler.cpp:194-217,256-272,
// window from :328-372). Slots are described by per-vx-row offsets instead of a 12-byte triple
// per slot, so the per-cycle upload stays a few KB.
void enumerate_axes(const kc_planner_config &c, const double vel[3], Axes &a) {
  int nx, ny;
  linear_split(c.control_type, c.max_linear_samples, nx, ny);
  const int nang = c.max_angular_samples + 1 - (c.max_angular_samples % 2);
  double vy_max = c.vy_max, vy_acc = c.vy_acc, vy_dec = c.vy_dec;
  if (c.control_type != KC_OMNI) vy_max = vy_acc = vy_dec = 0.0;  // trajectory_sampler.cpp:51-54
  const double ts = c.time_step;
  const double max_vx = std::min(c.vx_max, vel[0] + c.vx_acc * ts);
  const double min_vx = std::max(-c.vx_max, vel[0] - c.vx_dec * ts);
  double max_vy = 0.0, min_vy = 0.0;
  if (c.control_type == KC_OMNI) {
    max_vy = std::min(vy_max, vel[1] + vy_acc * ts);
    min_vy = std::max(-vy_max, vel[1] - vy_dec * ts);
  }
  const double res_x = std::max((max_vx - min_vx) / (nx - 1), 0.001);
  const double res_y = (ny > 1) ? std::max((max_vy - min_vy) / (ny - 1), 0.001) : 0.001;
  const double max_om = std::min(c.omega_max, vel[2] + c.omega_acc * ts);
  const double min_om = std::max(-c.omega_max, vel[2] - c.omega_dec * ts);
  const double res_om = std::max((max_om - min_om) / (nang - 1), 0.001);

  a.vx.clear();
  a.vy.clear();
  a.om.clear();
  a.row_off.clear();
  for (double om = min_om; om <= max_om; om += res_om) a.om.push_back(om);
  a.nom = (int32_t)a.om.size();
  const bool omni = c.control_type == KC_OMNI;
  if (omni)
    for (double vy = min_vy; vy <= max_vy; vy += res_y) a.vy.push_back(vy);
  a.nvy = (int32_t)a.vy.size();
  int32_t off = 0;
  double mvx = 0.0, mvy = 0.0;
  for (double vx = min_vx; vx <= max_vx; vx += res_x) {
    const bool arc = std::abs(vx) >= kMinVel;
    if (!omni && !arc) continue;  // non-holonomic: vx ~ 0 rows produce no slot
    a.vx.push_back(vx);
    a.row_off.push_back(off);
    off += a.nvy + (arc ? a.nom : 0);
    mvx = std::max(mvx, std::abs(vx));
  }
  a.row_off.push_back(off);
  a.n_slots = off;
  for (double vy : a.vy) mvy = std::max(mvy, std::abs(vy));
  a.max_speed = std::sqrt(mvx * mvx + mvy * mvy);
  // omni rows whose vx ~ 0 only carry the vy block; the decode relies on nvy + nom per arc row.
  // For those rows local >= nvy never happens because the row is exactly nvy long.
}

struct SensorDesc {
  int32_t is_cloud = 1;
  int32_t n = 0;
  const void *host = nullptr;  // scan: ranges then angles (two pointers handled by caller)
  const void *host2 = nullptr;
  const void *dev = nullptr;  // already-resident data (bank / batch), overrides host
};

}  // namespace

// robots per launch set of a batched sweep: workspace is sized for kBatchChunk, the default chunk is smaller
constexpr int kBatchChunk = 64;
constexpr int kBatchChunkDefault = 32;  // +1.6 % resident time against 64, finer upload / compute interleave when the host link is contended

struct kc_planner {
  kc_planner_config cfg;
  double base_horizon = 0.0, horizon = 0.0;
  int32_t P = 0;
  cudaStream_t stream = nullptr;
  // parallel branches of the cycle: k_path_cand (needs nothing), k_rollout_collide (needs the bitmap)
  cudaStream_t side = nullptr, side2 = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_fork2 = nullptr, ev_join2 = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::vector<cudaEvent_t> evk;
  int64_t launches = 0;
  hm::Rigid sensor_tf_body;

  // reference path
  DevBuf<float> d_path;  // X | Y | acc
  std::vector<float> hX, hY;
  int32_t path_n = 0;
  float path_len = 0.0f;

  // packed staging (ctx array | axes | sensor)
  PinnedBuf<uint8_t> h_stage;
  DevBuf<uint8_t> d_stage;

  // workspace (sized for R robots)
  DevBuf<uint32_t> d_zero;  // per robot: bitmap | cell_count | occ
  DevBuf<uint32_t> d_dil;   // per robot: k_dilate's two maps of the bitmap (2 x kDilMaxWords)
  DevBuf<uint32_t> d_sph;
  DevBuf<double2> d_tab_sc;      // heading table of the cycle: sincos per (omega row, step)
  DevBuf<float> d_tab_yaw;
  DevBuf<float2> d_bf_xy;        // brute-force verification hook: all sensor points, cost frame
  DevBuf<unsigned int> d_bf_min; // [2 x n_slots] FP32 / exact minima (float bits)
  DevBuf<float> d_bf_cost;
  DevBuf<int32_t> d_cell_start, d_cell_cursor, d_work_cells, d_pwork_cells;
  DevBuf<int2> d_tmp_cell;
  DevBuf<uint16_t> d_cell_nn, d_row_dx;
  DevBuf<int4> d_cell_info;
  DevBuf<float2> d_cand;
  DevBuf<int2> d_pcell_info;
  DevBuf<float2> d_pcand;
  DevBuf<int32_t> d_list, d_cutv;
  DevBuf<float> d_rowsxy;  // per robot: rows_x | rows_y of every slot (k_rollout_collide -> k_cost_eval)
  DevBuf<float2> d_tmp_xy, d_sorted_xy;
  DevBuf<float> d_costs;
  DevBuf<uint8_t> d_adm, d_prn;
  DevBuf<float> d_lbv, d_ubd;
  DevBuf<float2> d_sjv;
  DevBuf<int32_t> d_surv;
  DevBuf<unsigned long long> d_dmin, d_dbg;
  DevBuf<uint8_t> d_result;  // per robot: ResultHeader | rows
  PinnedBuf<uint8_t> h_result;
  // sampler mode
  DevBuf<float> d_rows, d_crows;
  DevBuf<int32_t> d_dst, d_cslots;
  PinnedBuf<uint8_t> h_samples;
  PinnedBuf<uint8_t> h_bulk;  // staging of large pageable uploads (upload_pageable)
  // evaluate mode
  DevBuf<float> d_in;
  DevBuf<int32_t> d_bbox;
  PinnedBuf<float> h_costs;
  PinnedBuf<uint8_t> h_adm;
  // setPointScan storage (CostEvaluator API)
  std::vector<uint8_t> cost_sensor;
  int32_t cost_sensor_is_cloud = 1, cost_sensor_n = 0;
  double cost_pose[3] = {0, 0, 0};
  float cost_D = 0.0f;
  // cloud bank (replay)
  DevBuf<float> d_bank;
  std::vector<int32_t> bank_counts;
  int32_t bank_slots = 0, bank_max = 0;
  // batch state kept resident for batch_replay
  int32_t batch_R = 0, batch_chunk = 0;  // robots of the resident batch / robots per launch set
  cudaStream_t copy = nullptr;           // H2D of the next chunk's clouds beside the running chunk
  cudaEvent_t ev_copy = nullptr;
  std::vector<RobotCtx> batch_ctx;
  std::vector<int> batch_starts;  // chunk boundaries of the resident batch (last entry = batch_R)
  int32_t batch_chunk_max = kBatchChunkDefault;  // tuning key 12: robots per launch set of a sweep (<= kBatchChunk)
  std::vector<int32_t> batch_chunk_P, batch_chunk_S;  // per chunk: largest P and tracked segment (launch geometry)
  int32_t batch_P = 0;        // largest P of the batch: stride of its result records
  bool batch_general = false;  // the batch's ctxs take the tilted-sensor rollout (scans through a tilted mount)
  DevBuf<float> d_batch_xyz;
  DevBuf<double> d_batch_scan;     // scans: per robot ranges | angles, in robot order
  PinnedBuf<double> h_batch_scan;  // their page-locked staging
  DevBuf<uint8_t> d_batch_stage;
  size_t batch_zero_words = 0, batch_sph_words = 0;
  int32_t batch_max_sensor = 0, batch_max_slots = 0, batch_max_qcells = 0, batch_dil_words = 0;
  // last cycle bookkeeping
  int32_t last_slots = 0;
  bool last_was_cycle = false;
  bool last_replay = false;  // the last cycle came from kc_planner_replay (ctx array, not d_stage[0])
  int32_t cand_cap = -1;  // tuning key 0 (-1: default)
  int cost_ctas_per_sm = 1, bounds_ctas_per_sm = 1;  // occupancy of k_cost_eval / k_cost_bounds (resident grids)
  // cached launch graph of one cycle (launch_cycle)
  struct GraphKey {
    const void *ctx, *zero, *sph;
    size_t zw, sw;
    int R, max_sensor, max_slots, P, S, mode, qcells, dil_words;
    bool any_points, heavy, general;
    bool operator==(const GraphKey &o) const {
      return ctx == o.ctx && zero == o.zero && sph == o.sph && zw == o.zw && sw == o.sw && R == o.R &&
             max_sensor == o.max_sensor && max_slots == o.max_slots && P == o.P && S == o.S &&
             mode == o.mode && qcells == o.qcells && dil_words == o.dil_words && any_points == o.any_points &&
             heavy == o.heavy && general == o.general;
    }
  };
  struct GraphSlot {
    GraphKey key{};
    cudaGraphExec_t exec = nullptr;
    int kernels = 0;
    uint64_t stamp = 0;
  };
  static constexpr int kGraphSlots = 160;  // e.g. one per resident cloud of a replay bank
  GraphSlot graphs[kGraphSlots];
  uint64_t graph_clock = 0;
  bool use_graphs = true;  // tuning key 1
  // tuning key 4: per-kernel CUDA events around every kernel of a plain-launch cycle (developer
  // timeline; kc_planner_debug_timeline reads them back)
  bool timeline = false;
  cudaEvent_t tl_ev[24] = {};
  int tl_n = 0;
  const char *tl_name[12] = {};
  // tuning key 7: branch and bound over the slots (k_cost_bounds): 0 off, 1 when the cycle has at
  // least kPruneMinSlots velocity slots (default; two more launches do not pay for fewer), 2 always
  int32_t use_prune = 1;
  bool prune_for(int32_t max_slots) const {
    return use_prune == 2 || (use_prune == 1 && max_slots >= 2048);
  }
  bool use_pdl = true;            // programmatic dependent launches on the bounds -> split -> eval chain
  // tuning key 10: disc size beyond which a candidate cell counts as heavy. -1 (default): kHeavyDefault
  // with the CTA-cooperative kernel launched only while the scene needs it - every cycle reports its
  // heavy-cell count in the result record, and the next cycle runs k_cell_cand_heavy iff the last
  // count was non-zero (scenes are coherent from one control cycle to the next; a first dense cycle
  // builds its heavy cells in place, as correct and slower). > 0: that threshold, kernel always on;
  // 0: never.
  int32_t heavy_points = -1;
  // tuning key 13: survivors of the bound stage up to which k_cost_eval spreads (slot, point) pairs over
  // the grid instead of handing whole slots to warps
  int32_t by_point_max = 2048;
  // tuning key 11: per-cell candidate lists. 1 (default): always built. -1: only when every slot is
  // evaluated exactly (no branch and bound); 0: never - exact queries then search their own disc
  // (warp_nn_search_one). Measured on B200 at config 2 (profiles/r2_family.json): without lists a cycle
  // whose bounds prune nearly everything gains 1-3 us, one with hundreds of survivors (clutter inside
  // reach) goes from 0.10 to 0.32 ms - the lists stay on.
  int32_t cand_lists = 1;
  bool heavy_seen = false;  // the last cycle whose result was read met heavy cells
  int32_t heavy_threshold() const { return heavy_points < 0 ? kHeavyDefault : heavy_points; }
  bool heavy_kernel_on() const { return heavy_points > 0 || (heavy_points < 0 && heavy_seen); }
  // the decision the CURRENT launch set was bound with (ctx.heavy_queue and the kernel list must agree;
  // taken once per call before the ctxs are filled, kept with a resident batch for its replays)
  bool heavy_bound = false, batch_heavy = false;
  // the launch set in flight runs the tilted-sensor instantiation of the rollout kernel (its ctxs have
  // coll_general set): scans through a pitched / rolled mount only; clouds arrive in the world frame
  bool general_bound = false;
  bool use_reach_mask = true;     // tuning key 5: candidate lists only for cells inside the analytic reach set
  bool zero_copy_cloud = true;    // tuning key 2: k_prep_points reads a page-locked caller cloud in place
  bool poll_result = true;        // tuning key 8: the host polls the mapped result record instead of a stream sync
  uint32_t cycle_seq = 0;
  bool mapped_result = true;      // tuning key 3: the winner record is written straight into pinned host memory
  RobotCtx last_ctx;      // device pointers of the last single-robot cycle (debug stats)
};

namespace {

struct Sizes {  // per-robot workspace requirements of one cycle
  size_t bitmap_words = 0, sph_words = 0;
  int32_t n_sensor = 0, n_slots = 0;
};

// sensor_tf_world_ -> the planar octree frame of the ctx, robot footprint bounds and row masks
// (ref: collision_check.h:91-136, collision_check.cpp:125-135)
int32_t fill_collision_frame(const kc_planner_config &c, const hm::Rigid &stw,
                             const hm::Rigid &sensor_tf_body, RobotCtx &cx) {
  cx.shape = c.robot_shape;
  cx.dim0 = (double)c.robot_dims[0];
  cx.dim1 = (double)c.robot_dims[1];
  cx.dim2 = (double)c.robot_dims[2];
  cx.res = c.octree_resolution;
  cx.res_factor = 1.0 / c.octree_resolution;
  const hm::Rot &L = stw.R;
  cx.a00 = L(0, 0);
  cx.a01 = L(0, 1);
  cx.a10 = L(1, 0);
  cx.a11 = L(1, 1);
  cx.tx = stw.t[0];
  cx.ty = stw.t[1];
  cx.tz = stw.t[2];
  const double tol = 1e-4;
  // the octree's z axis must stay vertical: upright, or upside down (a sensor flipped about x or y
  // keeps its voxel cubes axis-aligned with the upright robot solid; the xy block is then a
  // reflection). z_w = zsign * z_s + tz, so the robot centre (z_w = 0) sits at z_s = -zsign * tz.
  const double det = cx.a00 * cx.a11 - cx.a01 * cx.a10;
  const double zsign = (L(2, 2) >= 0.0f) ? 1.0 : -1.0;
  const bool planar = std::abs(L(0, 2)) < tol && std::abs(L(1, 2)) < tol &&
                      std::abs(L(2, 0)) < tol && std::abs(L(2, 1)) < tol &&
                      std::abs(std::abs((double)L(2, 2)) - 1.0) < tol &&
                      std::abs(cx.a00 * cx.a00 + cx.a10 * cx.a10 - 1.0) < 1e-3 &&
                      std::abs(std::abs(det) - 1.0) < 1e-3;
  cx.coll_general = 0;
  if (!planar) {
    // tilted mount (pitched lidar, depth camera): the octree's cubes are oriented boxes in the robot's
    // frame. The transform must be a rotation: unit quaternion within 1e-3 (the bound the parity checker uses too)
    bool orthonormal = true;
    for (int i = 0; i < 3 && orthonormal; ++i)
      for (int j = i; j < 3; ++j) {
        const double d = (double)L(0, i) * (double)L(0, j) + (double)L(1, i) * (double)L(1, j) +
                         (double)L(2, i) * (double)L(2, j);
        if (std::abs(d - (i == j ? 1.0 : 0.0)) > 1e-3) orthonormal = false;
      }
    KC_REQUIRE(orthonormal, KC_ERR_UNSUPPORTED,
               "collision checking needs a rotation as sensor_rotation (unit quaternion within 1e-3)");
    cx.coll_general = 1;
    for (int i = 0; i < 3; ++i) {
      for (int j = 0; j < 3; ++j) cx.gR[i * 3 + j] = (double)L(i, j);
      cx.gt[i] = (double)stw.t[i];
    }
  }
  cx.cz = -zsign * cx.tz;
  cx.sigma = (det >= 0.0) ? 1.0 : -1.0;
  cx.psi = std::atan2(cx.a10, cx.a00);
  if (c.robot_shape == KC_CYLINDER)
    cx.circ_r = cx.dim0;
  else if (c.robot_shape == KC_BOX)
    cx.circ_r = 0.5 * std::sqrt(cx.dim0 * cx.dim0 + cx.dim1 * cx.dim1);
  else
    cx.circ_r = cx.dim0;
  cx.scan_z = (float)(-(double)sensor_tf_body.t[2] / 2.0);
  // a voxel column touching the bounding circle of radius R around a pose in column k lies in
  // [k - floor(R/res) - 1, k + floor(R/res) + 1] (strictly inside (R/res + 1) columns of the
  // pose's own one); one more ring for the rounding of the division that finds k
  KC_REQUIRE(cx.circ_r / cx.res < 8192.0, KC_ERR_UNSUPPORTED,
             "octree_resolution %.6g is too fine for a robot of radius %.3f m", cx.res, cx.circ_r);
  cx.hit_W = (int32_t)std::floor(cx.circ_r / cx.res) + 2;
  cx.rho = (float)(cx.circ_r / cx.res);
  cx.use_rowmask = cx.hit_W <= 15 ? 1 : 0;
  if (cx.use_rowmask) {
    // a column at offset (dx, dy) is at least (max(|dx|-1,0), max(|dy|-1,0)) voxels away from a
    // pose anywhere inside its own voxel; the rounding of the division that finds the pose's
    // voxel moves that bound by ~1e-16 voxels, the limit below carries 1e-6
    const double lim = (cx.circ_r / cx.res) * (1.0 + 1e-6) + 1e-6;
    for (int dy = 0; dy <= cx.hit_W; ++dy) {
      uint32_t m = 0;
      for (int dx = -cx.hit_W; dx <= cx.hit_W; ++dx) {
        const double gx = std::max(std::abs(dx) - 1, 0), gy = std::max(dy - 1, 0);
        if (gx * gx + gy * gy <= lim * lim) m |= 1u << (dx + cx.hit_W);
      }
      cx.rowmask[dy] = m;
    }
    // the sure mask: a column at offset (dx, dy) is at most (|dx|, |dy|) voxels away from a pose anywhere
    // inside its own voxel; within the inscribed circle (cylinder: its radius; box: the shorter half
    // side, whatever the heading) with the FP32 filter's margins the exact test can only report a hit.
    // Spheres test a per-column height term as well: no shortcut.
    double rin = 0.0;
    if (c.robot_shape == KC_CYLINDER) rin = cx.dim0 / cx.res;
    if (c.robot_shape == KC_BOX) rin = 0.5 * std::min(cx.dim0, cx.dim1) / cx.res;
    const double lim2 = rin * rin * 0.9998 - 1e-6;
    for (int dy = 0; dy <= cx.hit_W; ++dy) {
      uint32_t m = 0;
      for (int dx = -cx.hit_W; dx <= cx.hit_W; ++dx)
        if ((double)(dx * dx + dy * dy) < lim2) m |= 1u << (dx + cx.hit_W);
      cx.suremask[dy] = m & cx.rowmask[dy];
    }
  }
  return KC_OK;
}

// bitmap window: every voxel column a pose inside the octree-frame box [x_lo, x_hi] x [y_lo, y_hi]
// can touch
// general (tilted) frames: every voxel a body centred within `reach` of the world point (wx, wy, 0) can
// touch, as a 3-D key window of the octree frame (a cube around the centre's image: conservative)
int32_t fill_collision_window_general(const kc_planner_config &c, double wx, double wy, double reach,
                                      RobotCtx &cx, Sizes &sz) {
  double rho;
  if (c.robot_shape == KC_SPHERE)
    rho = cx.dim0;
  else if (c.robot_shape == KC_CYLINDER)
    rho = std::sqrt(cx.dim0 * cx.dim0 + 0.25 * cx.dim1 * cx.dim1);
  else
    rho = 0.5 * std::sqrt(cx.dim0 * cx.dim0 + cx.dim1 * cx.dim1 + cx.dim2 * cx.dim2);
  const double d[3] = {wx - cx.gt[0], wy - cx.gt[1], 0.0 - cx.gt[2]};
  const double E = reach + rho + 2.0 * cx.res + 1e-3;
  double lo[3], hi[3];
  for (int j = 0; j < 3; ++j) {
    const double cs = cx.gR[0 * 3 + j] * d[0] + cx.gR[1 * 3 + j] * d[1] + cx.gR[2 * 3 + j] * d[2];
    lo[j] = std::floor((cs - E) / cx.res) - 2;
    hi[j] = std::floor((cs + E) / cx.res) + 2;
    KC_REQUIRE(std::abs(lo[j]) < 1e9 && hi[j] - lo[j] < 4096, KC_ERR_UNSUPPORTED,
               "octree_resolution %.6g is too fine for a tilted sensor and poses spread over %.3f m "
               "(voxel window > 4096 per axis)", cx.res, 2 * E);
  }
  cx.g_kx0 = (int32_t)lo[0];
  cx.g_ky0 = (int32_t)lo[1];
  cx.g_kz0 = (int32_t)lo[2];
  cx.g_nx = (int32_t)(hi[0] - lo[0]) + 1;
  cx.g_ny = (int32_t)(hi[1] - lo[1]) + 1;
  cx.g_nz = (int32_t)(hi[2] - lo[2]) + 1;
  cx.g_wpr = (cx.g_nx + 31) / 32;
  const double words = (double)cx.g_nz * cx.g_ny * cx.g_wpr;
  KC_REQUIRE(words < 64.0 * 1024 * 1024, KC_ERR_UNSUPPORTED,
             "octree_resolution %.6g is too fine for a tilted sensor: the voxel window would need %.0f MB",
             cx.res, words * 4 / 1e6);
  cx.bm_kx0 = cx.bm_ky0 = 0;
  cx.bm_cols = cx.bm_rows = cx.bm_wpr = 0;
  sz.bitmap_words = (size_t)words;
  sz.sph_words = 0;
  return KC_OK;
}

int32_t fill_collision_window(const kc_planner_config &c, double x_lo, double x_hi, double y_lo,
                              double y_hi, RobotCtx &cx, Sizes &sz) {
  const double E = cx.circ_r + 2.0 * cx.res + 1e-3;
  const double kx_lo = std::floor((x_lo - E) / cx.res) - 1, kx_hi = std::floor((x_hi + E) / cx.res) + 1;
  const double ky_lo = std::floor((y_lo - E) / cx.res) - 1, ky_hi = std::floor((y_hi + E) / cx.res) + 1;
  KC_REQUIRE(std::abs(kx_lo) < 1e9 && std::abs(ky_lo) < 1e9 && kx_hi - kx_lo < 16384 &&
                 ky_hi - ky_lo < 16384,
             KC_ERR_UNSUPPORTED,
             "octree_resolution %.6g is too fine for poses spread over %.3f x %.3f m (voxel window > 16384)",
             cx.res, x_hi - x_lo + 2 * E, y_hi - y_lo + 2 * E);
  cx.bm_kx0 = (int32_t)kx_lo;
  cx.bm_ky0 = (int32_t)ky_lo;
  cx.bm_cols = (int32_t)(kx_hi - kx_lo) + 1;
  cx.bm_rows = (int32_t)(ky_hi - ky_lo) + 1;
  cx.bm_wpr = (cx.bm_cols + 31) / 32;
  sz.bitmap_words = (size_t)cx.bm_rows * cx.bm_wpr;
  sz.sph_words = 0;
  if (c.robot_shape == KC_SPHERE) sz.sph_words = (size_t)cx.bm_rows * cx.bm_cols;
  return KC_OK;
}

// the planner's own reference path (kc_planner_set_path), as the single-robot entry points use it
BatchPath own_path(const kc_planner *p) {
  BatchPath b;
  b.hX = p->hX.data();
  b.hY = p->hY.data();
  b.dX = p->d_path.ptr;
  b.dY = p->d_path.ptr + p->path_n;
  b.dAcc = p->d_path.ptr + 2 * (size_t)p->path_n;
  b.n = p->path_n;
  b.total_length = p->path_len;
  return b;
}

// Fill everything of the ctx that does not depend on device pointers. Returns KC_OK or an error.
// P: points per trajectory of this robot; path: its reference path.
int32_t fill_ctx_scalars(kc_planner *p, int32_t P, const BatchPath &path, const double vel[3],
                         const double pose[3], const SensorDesc &sd, int32_t seg_start, int32_t seg_count,
                         bool want_coll, bool want_cost, float D, const double cost_pose[3], const Axes &ax,
                         RobotCtx &cx, Sizes &sz) {
  const kc_planner_config &c = p->cfg;
  memset(&cx, 0, sizeof(cx));
  cx.pose_x = pose[0];
  cx.pose_y = pose[1];
  cx.pose_yaw = pose[2];
  cx.dt = (double)(float)c.time_step;
  cx.P = P;
  cx.n_slots = ax.n_slots;
  cx.n_rows = (int32_t)ax.vx.size();
  cx.nvy = ax.nvy;
  cx.nom = ax.nom;
  cx.drop_samples = c.drop_samples;
  cx.num_ctrl_points = c.num_ctrl_points;
  cx.sensor_is_cloud = sd.is_cloud;
  cx.n_sensor = sd.n;
  sz.n_sensor = sd.n;
  sz.n_slots = ax.n_slots;

  const double reach = ax.max_speed * (double)(P - 1) * cx.dt * 1.001 + 1e-3;

  // ---- collision world (ref: collision_check.h:91-136, collision_check.cpp:125-135) ----
  cx.coll_enabled = (want_coll && sd.n > 0) ? 1 : 0;
  cx.shape = c.robot_shape;
  cx.dim0 = (double)c.robot_dims[0];
  cx.dim1 = (double)c.robot_dims[1];
  cx.dim2 = (double)c.robot_dims[2];
  cx.res = c.octree_resolution;
  cx.res_factor = 1.0 / c.octree_resolution;
  if (want_coll) {
    hm::Rigid stw;  // sensor_tf_world_
    if (sd.is_cloud) {
      const float q[4] = {0, 0, 0, 1}, t[3] = {0, 0, 0};
      stw = hm::rigid_from_quat(q, t);  // global_frame = true -> identity (collision_check.h:121-123)
    } else {
      stw = hm::compose(hm::rigid_from_state(pose[0], pose[1], pose[2]), p->sensor_tf_body);
    }
    KC_TRY(fill_collision_frame(c, stw, p->sensor_tf_body, cx));
    // window of voxel columns any pose of this cycle can touch, in the octree frame
    if (cx.coll_general) {
      KC_TRY(fill_collision_window_general(c, (double)(float)pose[0], (double)(float)pose[1], reach, cx, sz));
    } else {
      const double dx = (double)(float)pose[0] - cx.tx, dy = (double)(float)pose[1] - cx.ty;
      const double c0x = cx.a00 * dx + cx.a10 * dy, c0y = cx.a01 * dx + cx.a11 * dy;
      KC_TRY(fill_collision_window(c, c0x - reach, c0x + reach, c0y - reach, c0y + reach, cx, sz));
    }
  }

  // ---- cost evaluator scalars ----
  {
    // ref: cost_evaluator.h:180,189: sensor_tf_body_ * body_tf_world_ (operand order as written)
    const hm::Rigid T =
        hm::compose(p->sensor_tf_body, hm::rigid_from_state(cost_pose[0], cost_pose[1], cost_pose[2]));
    for (int i = 0; i < 9; ++i) cx.T[i] = T.R.r[i];
    cx.T[9] = T.t[0];
    cx.T[10] = T.t[1];
    cx.T[11] = T.t[2];
  }
  cx.D = D;
  cx.w_path = c.w_path;
  cx.w_goal = c.w_goal;
  cx.w_obs = c.w_obstacles;
  cx.w_smooth = c.w_smooth;
  cx.w_jerk = c.w_jerk;
  cx.acc0 = (float)c.vx_acc;  // ref: cost_evaluator.cpp:18-20
  cx.acc1 = (float)c.vy_acc;
  cx.acc2 = (float)c.omega_acc;
  cx.obs_enabled = (want_cost && sd.n > 0 && c.w_obstacles > 0.0) ? 1 : 0;
  cx.path_enabled = (want_cost && path.total_length > 0.0f) ? 1 : 0;
  cx.path_n = path.n;
  cx.path_len = path.total_length;
  cx.seg_start = 0;
  cx.seg_count = 0;
  if (want_cost) {
    // ref: path.cpp:80-86 Path::getPart range check
    KC_REQUIRE(seg_start >= 0 && seg_count >= 1 && seg_start + seg_count <= path.n,
               KC_ERR_OUT_OF_RANGE,
               "Invalid range for path part. Maximum path size is %d, but requested part start= "
               "%d, and requested end= %d",
               path.n, seg_start, seg_start + seg_count - 1);
    cx.seg_start = seg_start;
    cx.seg_count = seg_count;
    // ref: path.h:85-91 View::totalSegmentLength (float sum of float norms, index order)
    float len = 0.0f;
    for (int i = 0; i + 1 < seg_count; ++i) {
      const float ddx = path.hX[seg_start + i] - path.hX[seg_start + i + 1];
      const float ddy = path.hY[seg_start + i] - path.hY[seg_start + i + 1];
      len += std::sqrt(ddx * ddx + (ddy * ddy + 0.0f));
    }
    cx.seg_len = len;
    double step = 0.0;
    for (int i = 0; i + 1 < seg_count; ++i)
      step = std::max(step, std::hypot((double)path.hX[seg_start + i] - (double)path.hX[seg_start + i + 1],
                                       (double)path.hY[seg_start + i] - (double)path.hY[seg_start + i + 1]));
    cx.seg_step = (float)(step * (1.0 + 1e-6) + 1e-9);
    if (!(cx.seg_step < 1e30f)) cx.seg_step = 1e30f;  // non-finite path: disables the pruning
  }
  cx.dcap2 = (double)D * (double)D * (1.0 + 1e-5) + 1e-12;
  // analytic reach set of this cycle's velocity window (see cell_reachable); non-holonomic only
  cx.reach_mask = 0;
  if (p->use_reach_mask && want_coll && want_cost && c.control_type != KC_OMNI && ax.n_slots > 0 &&
      P >= 4 && !ax.vx.empty() && !ax.om.empty()) {
    double vf = 0.0, vr = 0.0, om_lo = ax.om.front(), om_hi = ax.om.front();
    for (double v : ax.vx) {
      vf = std::max(vf, v);
      vr = std::max(vr, -v);
    }
    for (double o : ax.om) {
      om_lo = std::min(om_lo, o);
      om_hi = std::max(om_hi, o);
    }
    const int n = P - 2;
    cx.reach_mask = 1;
    cx.rm_n = n;
    cx.rm_px = (float)pose[0];
    cx.rm_py = (float)pose[1];
    cx.rm_yaw = (float)pose[2];
    cx.rm_vf = (float)(vf * cx.dt * 1.001);
    cx.rm_vr = (float)(vr * cx.dt * 1.001);
    cx.rm_blo = (float)(std::min(om_lo, 0.0) * cx.dt * 0.5 * n * 1.001 - 1e-3);
    cx.rm_bhi = (float)(std::max(om_hi, 0.0) * cx.dt * 0.5 * n * 1.001 + 1e-3);
  }
  return KC_OK;
}

// obstacle-grid window: square centred on (cxw, cyw) with half extent `half`
// qhalf: half extent of the square (around the same centre) that can contain trajectory points
void set_grid_window(RobotCtx &cx, float cxw, float cyw, double half, double qhalf) {
  cx.win_lo_x = (float)((double)cxw - half);
  cx.win_hi_x = (float)((double)cxw + half);
  cx.win_lo_y = (float)((double)cyw - half);
  cx.win_hi_y = (float)((double)cyw + half);
  cx.gx0 = cx.win_lo_x;
  cx.gy0 = cx.win_lo_y;
  const double span = std::max((double)cx.win_hi_x - cx.win_lo_x, (double)cx.win_hi_y - cx.win_lo_y);
  cx.h = (float)(span / kGridN * (1.0 + 1e-6));
  cx.inv_h = 1.0f / cx.h;
  const double ih = 1.0 / (double)cx.h;
  cx.q_x0 = std::max(0, (int)std::floor(((double)cxw - qhalf - cx.gx0) * ih) - 1);
  cx.q_x1 = std::min(kGridN - 1, (int)std::floor(((double)cxw + qhalf - cx.gx0) * ih) + 1);
  cx.q_y0 = std::max(0, (int)std::floor(((double)cyw - qhalf - cx.gy0) * ih) - 1);
  cx.q_y1 = std::min(kGridN - 1, (int)std::floor(((double)cyw + qhalf - cx.gy0) * ih) + 1);
}

inline int32_t qcells(const RobotCtx &cx) {
  return std::max(0, cx.q_x1 - cx.q_x0 + 1) * std::max(0, cx.q_y1 - cx.q_y0 + 1);
}

constexpr size_t kDilMaxWords = 4096;  // largest bitmap (words) k_dilate derives its maps for
// per-robot zero-initialised region: bitmap | best_key | counters | blk_tot | occ | cell_count
constexpr size_t kTailWords = (size_t)kGridN * kGridN + 1 + (size_t)kGridN * kGridWords + kScanBlocks + 16;
constexpr int32_t kCandCap = 1 << 19;  // candidate pool entries per robot (4 MB); overflow -> generic search
constexpr int32_t kPathCandCap = 1 << 19;  // same for the tracked-segment candidates (path cost)
size_t zero_words_per_robot(size_t bitmap_words) {
  return align_up(((bitmap_words + 1) / 2 * 2 + kTailWords) * 4) / 4;
}

// heading table: one row per omega of the axis plus the omega = 0 row of the omni vy block
inline int table_rows_max(const kc_planner_config &c) {
  return c.max_angular_samples + 1 - (c.max_angular_samples % 2) + 1;
}
inline int table_ctas(const kc_planner_config &c) { return (table_rows_max(c) + 7) / 8; }  // 8 warps per CTA

// carve per-robot workspace pointers
int32_t reserve_workspace(kc_planner *p, int R, size_t zero_words, size_t sph_words, int32_t max_sensor,
                          int32_t max_slots, int32_t P) {
  KC_TRY(p->d_zero.reserve((size_t)R * zero_words));
  KC_TRY(p->d_dil.reserve((size_t)R * 2 * kDilMaxWords));
  KC_TRY(p->d_tab_sc.reserve((size_t)R * table_rows_max(p->cfg) * std::max(P - 1, 1)));
  KC_TRY(p->d_tab_yaw.reserve((size_t)R * table_rows_max(p->cfg) * std::max(P - 1, 1)));
  if (sph_words) KC_TRY(p->d_sph.reserve((size_t)R * sph_words));
  KC_TRY(p->d_cell_start.reserve((size_t)R * (kGridN * kGridN + 1)));
  KC_TRY(p->d_cell_cursor.reserve((size_t)R * kGridN * kGridN));
  KC_TRY(p->d_work_cells.reserve((size_t)R * kGridN * kGridN));
  KC_TRY(p->d_pwork_cells.reserve((size_t)R * kGridN * kGridN));
  KC_TRY(p->d_cell_nn.reserve((size_t)R * kGridN * kGridN));
  KC_TRY(p->d_row_dx.reserve((size_t)R * kGridN * kGridN));
  KC_TRY(p->d_cell_info.reserve((size_t)R * kGridN * kGridN));
  KC_TRY(p->d_cand.reserve((size_t)R * kCandCap));
  KC_TRY(p->d_pcell_info.reserve((size_t)R * kGridN * kGridN));
  KC_TRY(p->d_pcand.reserve((size_t)R * kPathCandCap));
  KC_TRY(p->d_tmp_cell.reserve((size_t)R * std::max(max_sensor, 1)));
  KC_TRY(p->d_tmp_xy.reserve((size_t)R * std::max(max_sensor, 1)));
  KC_TRY(p->d_sorted_xy.reserve((size_t)R * std::max(max_sensor, 1)));
  KC_TRY(p->d_costs.reserve((size_t)R * std::max(max_slots, 1)));
  KC_TRY(p->d_adm.reserve((size_t)R * std::max(max_slots, 1)));
  KC_TRY(p->d_prn.reserve((size_t)R * std::max(max_slots, 1)));
  KC_TRY(p->d_lbv.reserve((size_t)R * std::max(max_slots, 1)));
  KC_TRY(p->d_ubd.reserve((size_t)R * std::max(max_slots, 1)));
  KC_TRY(p->d_sjv.reserve((size_t)R * std::max(max_slots, 1)));
  KC_TRY(p->d_surv.reserve((size_t)R * std::max(max_slots, 1)));
  KC_TRY(p->d_dmin.reserve((size_t)R * std::max(max_slots, 1)));
  KC_TRY(p->d_dbg.reserve(96));
  KC_TRY(p->d_list.reserve((size_t)R * std::max(max_slots, 1)));
  KC_TRY(p->d_cutv.reserve((size_t)R * std::max(max_slots, 1)));
  KC_TRY(p->d_rowsxy.reserve((size_t)R * std::max(max_slots, 1) * P * 2));
  const size_t res_bytes = align_up(sizeof(ResultHeader) + sizeof(float) * (5 * (size_t)P));
  KC_TRY(p->d_result.reserve((size_t)R * res_bytes));
  KC_TRY(p->h_result.reserve((size_t)R * res_bytes));
  return KC_OK;
}

// r: workspace slot of this robot; r_result: slot of its result record (the batch reuses the
// workspace chunk after chunk but keeps one result record per robot). P: the launch set's largest
// points per trajectory, which sizes the per-robot strides (a robot's own cx.P may be smaller).
void bind_workspace(kc_planner *p, RobotCtx &cx, const BatchPath &path, int r, size_t zero_words,
                    size_t bitmap_words, size_t sph_words, int32_t max_sensor, int32_t max_slots, int32_t P,
                    int r_result = -1) {
  uint32_t *z = p->d_zero.ptr + (size_t)r * zero_words;
  {
    const size_t stride = (size_t)table_rows_max(p->cfg) * std::max(P - 1, 1);
    cx.tab_sc = p->d_tab_sc.ptr + (size_t)r * stride;
    cx.tab_yaw = p->d_tab_yaw.ptr + (size_t)r * stride;
    cx.tab_rows = (cx.n_slots > 0) ? cx.nom + 1 : 0;
    cx.tab_ctas = (cx.n_slots > 0) ? table_ctas(p->cfg) : 0;
  }
  cx.bitmap = z;
  cx.dil_maps = p->d_dil.ptr + (size_t)r * 2 * kDilMaxWords;
  cx.dil_stride = (int32_t)kDilMaxWords;
  uint32_t *q = z + (bitmap_words + 1) / 2 * 2;  // keep 8-byte alignment for best_key
  cx.best_key = reinterpret_cast<unsigned long long *>(q);
  cx.done_ctr = q + 2;
  cx.adm_count = reinterpret_cast<int32_t *>(q + 3);
  cx.cand_ctr = reinterpret_cast<int32_t *>(q + 4);
  cx.pcand_ctr = reinterpret_cast<int32_t *>(q + 5);
  cx.heavy_ctr = reinterpret_cast<int32_t *>(q + 10);
  cx.heavy_points = p->heavy_threshold();
  cx.by_point_max = p->by_point_max;
  cx.heavy_queue = p->heavy_bound ? 1 : 0;
  cx.cand_lists = (p->cand_lists == 1 || (p->cand_lists < 0 && !p->prune_for(max_slots))) ? 1 : 0;
  cx.pcell_info = p->d_pcell_info.ptr + (size_t)r * kGridN * kGridN;
  cx.pcand_pool = p->d_pcand.ptr + (size_t)r * kPathCandCap;
  cx.pcand_cap = (p->cand_cap >= 0) ? std::min(p->cand_cap, kPathCandCap) : kPathCandCap;
  // cycles evaluate the path cost from per-cell candidate lists of the tracked segment
  // (k_path_cand); the CostEvaluator entry point (caller-provided rows) keeps the direct search
  cx.pcand_enabled = (cx.path_enabled && cx.w_path > 0.0 && cx.n_slots > 0 && qcells(cx) > 0) ? 1 : 0;
  cx.bounds_done = q + 8;
  cx.n_surv = reinterpret_cast<int32_t *>(q + 9);
  cx.blk_tot = q + 16;  // 16 header words (kTailWords)
  cx.occ = q + 16 + kScanBlocks;
  cx.cell_count = reinterpret_cast<int32_t *>(q + 16 + kScanBlocks + (size_t)kGridN * kGridWords);
  cx.sph_col = sph_words ? p->d_sph.ptr + (size_t)r * sph_words : nullptr;
  cx.cell_start = p->d_cell_start.ptr + (size_t)r * (kGridN * kGridN + 1);
  cx.cell_cursor = p->d_cell_cursor.ptr + (size_t)r * kGridN * kGridN;
  cx.work_cells = p->d_work_cells.ptr + (size_t)r * kGridN * kGridN;
  cx.work_ctr = reinterpret_cast<int32_t *>(q + 11);
  cx.pwork_cells = p->d_pwork_cells.ptr + (size_t)r * kGridN * kGridN;
  cx.pwork_ctr = reinterpret_cast<int32_t *>(q + 12);
  cx.cell_nn = p->d_cell_nn.ptr + (size_t)r * kGridN * kGridN;
  cx.row_dx = p->d_row_dx.ptr + (size_t)r * kGridN * kGridN;
  cx.cell_info = p->d_cell_info.ptr + (size_t)r * kGridN * kGridN;
  cx.cand_pool = p->d_cand.ptr + (size_t)r * kCandCap;
  cx.cand_cap = (p->cand_cap >= 0) ? std::min(p->cand_cap, kCandCap) : kCandCap;
  const size_t ms = (size_t)std::max(max_sensor, 1), msl = (size_t)std::max(max_slots, 1);
  cx.tmp_cell = p->d_tmp_cell.ptr + r * ms;
  cx.tmp_xy = p->d_tmp_xy.ptr + r * ms;
  cx.sorted_xy = p->d_sorted_xy.ptr + r * ms;
  cx.costs = p->d_costs.ptr + r * msl;
  cx.adm = p->d_adm.ptr + r * msl;
  cx.prn = p->d_prn.ptr + r * msl;
  cx.lbv = p->d_lbv.ptr + r * msl;
  cx.ubd = p->d_ubd.ptr + r * msl;
  cx.sjv = p->d_sjv.ptr + r * msl;
  cx.surv = p->d_surv.ptr + r * msl;
  cx.dmin_bits = p->d_dmin.ptr + r * msl;
  cx.dbg = p->d_dbg.ptr;
  cx.ub_inv = q + 7;
  cx.prune = p->prune_for(max_slots) ? 1 : 0;
  cx.list = p->d_list.ptr + r * msl;
  cx.cutv = p->d_cutv.ptr + r * msl;
  cx.rows_x = p->d_rowsxy.ptr + r * msl * P * 2;
  cx.rows_y = cx.rows_x + msl * P;
  cx.n_list = reinterpret_cast<int32_t *>(q + 6);
  const size_t res_bytes = align_up(sizeof(ResultHeader) + sizeof(float) * (5 * (size_t)P));
  uint8_t *rb = p->d_result.ptr + (size_t)(r_result >= 0 ? r_result : r) * res_bytes;
  cx.result = reinterpret_cast<ResultHeader *>(rb);
  cx.res_rows = reinterpret_cast<float *>(rb + sizeof(ResultHeader));
  cx.pathX = path.dX;
  cx.pathY = path.dY;
  cx.pathAcc = path.dAcc;
}

int pick_eval_warps(int P, int S, int dil_words, size_t &smem) {  // k_eval_rows
  int warps = kEvalWarps;
  while (warps > 1 && eval_smem_bytes(P, S, warps, dil_words) > 200 * 1024) warps >>= 1;
  smem = eval_smem_bytes(P, S, warps, dil_words);
  return warps;
}
int pick_rollout_warps(int P, int dil_words, size_t &smem) {  // k_rollout_collide
  int warps = kEvalWarps;
  while (warps > 1 && rollout_smem_bytes(P, warps, dil_words) > 200 * 1024) warps >>= 1;
  smem = rollout_smem_bytes(P, warps, dil_words);
  return warps;
}
int pick_cost_warps(int P, int S, size_t &smem) {  // k_cost_eval
  int warps = kEvalWarps;
  while (warps > 1 && cost_smem_bytes(P, S, warps) > 200 * 1024) warps >>= 1;
  smem = cost_smem_bytes(P, S, warps);
  return warps;
}

// Dilated-bitmap precheck of the collision test (block_dilate_bitmap): enabled when the bitmap of
// the reachable window fits a CTA's shared memory; returns the words to reserve (0: disabled).
int32_t plan_dilation(RobotCtx &cx, size_t bitmap_words) {
  cx.dil_W = 0;
  if (!cx.coll_enabled || cx.coll_general || bitmap_words == 0 || bitmap_words > kDilMaxWords) return 0;
  const double w = (double)cx.hit_W;
  if (!(w >= 1.0 && w <= 31.0)) return 0;
  cx.dil_W = (int32_t)w;
  return (int32_t)bitmap_words;
}

// launch behind the previous kernel of the stream; pdl: as a programmatic dependent (the kernel's
// prologue overlaps the tail of its producer, see grid_dep_wait)
template <typename K>
void launch_after(K kernel, dim3 grid, int block, size_t smem, cudaStream_t st, const RobotCtx *ctx, bool pdl) {
  cudaLaunchConfig_t lc = {};
  lc.gridDim = grid;
  lc.blockDim = dim3(block);
  lc.dynamicSmemBytes = smem;
  lc.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  lc.attrs = at;
  lc.numAttrs = pdl ? 1 : 0;
  cudaLaunchKernelEx(&lc, kernel, ctx);
}

template <typename K>
int32_t allow_smem(K kernel, size_t smem) {
  if (smem > 48 * 1024) {
    KC_REQUIRE(smem <= 227 * 1024, KC_ERR_UNSUPPORTED,
               "trajectory too long for on-chip staging (%zu bytes of shared memory needed)", smem);
    KC_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  return KC_OK;
}

// enqueue the kernels of one cycle for R robots whose ctxs are at d_ctx; returns the kernel count.
//
//   main   memset -> k_prep_points -> k_scan_dist -> k_scatter (+ cell classification) -> k_cell_cand
//                                     [-> k_cell_cand_heavy] --+-> k_cost_bounds -> k_cost_split -> k_cost_eval
//   side   (after memset)  k_path_class -> k_path_cand -------/|
//   side2  (after k_prep_points)  k_dilate -> k_rollout_collide/
//
// With events requested (bench.py's kernel timing) the two trajectory kernels run on the main stream
// between the events instead, so that the events bracket exactly their work.
int32_t enqueue_cycle(kc_planner *p, const RobotCtx *d_ctx, int R, size_t zero_words_total,
                      size_t sph_words_total, int32_t max_sensor, int32_t max_slots, int P, int S,
                      bool any_points, int mode /*0 cycle, 1 sampler*/, cudaEvent_t eval_start,
                      cudaEvent_t eval_stop, int32_t max_qcells, int32_t dil_words, int &n_kernels) {
  cudaStream_t st = p->stream;
  n_kernels = 0;
  const bool timed = eval_start || eval_stop;
  p->tl_n = 0;
  // developer timeline: an event before and after each kernel, on the stream it runs on
  auto mark = [&](cudaStream_t q, const char *name, bool begin) {
    if (!p->timeline || p->tl_n >= 12) return;
    const int i = 2 * p->tl_n + (begin ? 0 : 1);
    if (!p->tl_ev[i]) cudaEventCreate(&p->tl_ev[i]);
    cudaEventRecord(p->tl_ev[i], q);
    if (begin)
      p->tl_name[p->tl_n] = name;
    else
      p->tl_n += 1;
  };
  mark(st, "memset", true);
  if (any_points || max_slots > 0) KC_CUDA(cudaMemsetAsync(p->d_zero.ptr, 0, zero_words_total * 4, st));
  mark(st, "memset", false);
  const bool path_branch = mode == 0 && max_slots > 0 && max_qcells > 0;
  if (path_branch) {
    KC_CUDA(cudaEventRecord(p->ev_fork, st));
    KC_CUDA(cudaStreamWaitEvent(p->side, p->ev_fork, 0));
    mark(p->side, "k_path_cand", true);
    k_path_class<<<dim3((max_qcells + 255) / 256, R), 256, 0, p->side>>>(d_ctx);
    k_path_cand<<<dim3((max_qcells + kCandWarps - 1) / kCandWarps, R), kCandWarps * 32, 0, p->side>>>(d_ctx);
    mark(p->side, "k_path_cand", false);
    KC_CUDA(cudaEventRecord(p->ev_join, p->side));
    n_kernels += 2;
  }
  size_t smem_r = 0, smem_c = 0;
  const int warps_r = pick_rollout_warps(P, dil_words, smem_r);
  const int warps_c = pick_cost_warps(P, S, smem_c);
  // resident grids of the cost kernels (one set of CTAs for a single robot, four sets shared by a
  // batch), each from its own kernel's occupancy
  auto resident_grid = [&](int ctas_per_sm) {
    const int cap = std::max(1, ctas_per_sm) * sm_count();
    const int want = (R == 1) ? cap : std::max(1, (4 * cap + R - 1) / R);
    return std::max(1, std::min((max_slots + warps_c - 1) / warps_c, want));
  };
  const int gx_cost = resident_grid(p->cost_ctas_per_sm), gx_bounds = resident_grid(p->bounds_ctas_per_sm);
  bool path_joined = false;
  auto launch_rollout = [&](cudaStream_t q) -> int32_t {
    const int tiles = (max_slots + kTileSlots - 1) / kTileSlots;  // one warp per tile of slots
    const dim3 grid((tiles + warps_r - 1) / warps_r, R);
    bool pdl = false;
    if (dil_words > 0) {  // the bitmap's derived maps, once per robot; the rollout's kinematics run beside it
      mark(q, "k_dilate", true);
      k_dilate<<<dim3((dil_words + 255) / 256, R), 256, 0, q>>>(d_ctx);
      mark(q, "k_dilate", false);
      n_kernels += 1;
      pdl = p->use_pdl && !p->timeline;
    }
    mark(q, "k_rollout_collide", true);
    if (mode == 0) {
      if (p->general_bound)
        launch_after(k_rollout_collide<false, true>, grid, warps_r * 32, smem_r, q, d_ctx, pdl);
      else
        launch_after(k_rollout_collide<false, false>, grid, warps_r * 32, smem_r, q, d_ctx, pdl);
    } else {
      if (p->general_bound)
        launch_after(k_rollout_collide<true, true>, grid, warps_r * 32, smem_r, q, d_ctx, pdl);
      else
        launch_after(k_rollout_collide<true, false>, grid, warps_r * 32, smem_r, q, d_ctx, pdl);
    }
    mark(q, "k_rollout_collide", false);
    n_kernels += 1;
    return KC_OK;
  };
  bool rollout_branch = false;
  if (any_points || max_slots > 0) {
    if (sph_words_total) KC_CUDA(cudaMemsetAsync(p->d_sph.ptr, 0xFF, sph_words_total * 4, st));
    const int gx = std::max(1, std::min((max_sensor + 255) / 256, 8 * sm_count()));
    const int tc = max_slots > 0 ? table_ctas(p->cfg) : 0;  // heading table for the rollouts
    mark(st, "k_prep_points", true);
    k_prep_points<<<dim3(gx + tc, R), 256, 0, st>>>(d_ctx);
    mark(st, "k_prep_points", false);
    n_kernels += 1;
  }
  if (any_points) {
    const int gx = std::max(1, std::min((max_sensor + 255) / 256, 8 * sm_count()));
    if (mode == 0) {
      if (max_slots > 0 && !timed) {  // rollouts need the bitmap only: beside the grid preparation
        rollout_branch = true;
        KC_CUDA(cudaEventRecord(p->ev_fork2, st));
        KC_CUDA(cudaStreamWaitEvent(p->side2, p->ev_fork2, 0));
        KC_TRY(launch_rollout(p->side2));
        KC_CUDA(cudaEventRecord(p->ev_join2, p->side2));
      }
      mark(st, "k_scan_dist", true);
      k_scan_dist<<<dim3(kScanBlocks, R), 1024, 0, st>>>(d_ctx);
      mark(st, "k_scan_dist", false);
      mark(st, "k_scatter", true);
      const int n_class = class_ctas_for(max_qcells);  // CTAs that classify the query-window cells
      k_scatter<<<dim3(gx + n_class, R), 256, 0, st>>>(d_ctx, n_class);
      mark(st, "k_scatter", false);
      n_kernels += 2;
      if (max_qcells > 0) {
        mark(st, "k_cell_cand", true);
        k_cell_cand<<<dim3((max_qcells + kCandWarps - 1) / kCandWarps, R), kCandWarps * 32, 0, st>>>(d_ctx);
        mark(st, "k_cell_cand", false);
        n_kernels += 1;
        if (p->heavy_bound) {  // cells next to dense clusters, one CTA each
          const int gh = (R == 1) ? 8 * sm_count() : std::max(8, (8 * sm_count() + R - 1) / R);
          mark(st, "k_cell_heavy", true);
          launch_after(k_cell_cand_heavy, dim3(gh, R), kHeavyThreads, 0, st, d_ctx, p->use_pdl && !p->timeline);
          mark(st, "k_cell_heavy", false);
          n_kernels += 1;
        }
      }
    }
  }
  if (max_slots > 0) {
    if (path_branch && !path_joined) {
      KC_CUDA(cudaStreamWaitEvent(st, p->ev_join, 0));
      path_joined = true;
    }
    if (eval_start) KC_CUDA(cudaEventRecord(eval_start, st));
    if (rollout_branch)
      KC_CUDA(cudaStreamWaitEvent(st, p->ev_join2, 0));
    else
      KC_TRY(launch_rollout(st));
    if (mode == 0) {
      const int gxc = gx_cost;
      if (p->prune_for(max_slots)) {  // stage 1 of the branch and bound: cheap terms + bounds of every slot
        mark(st, "k_cost_bounds", true);
        k_cost_bounds<<<dim3(gx_bounds, R), warps_c * 32, smem_c, st>>>(d_ctx);
        mark(st, "k_cost_bounds", false);
        launch_after(k_cost_split, dim3((max_slots + 255) / 256, R), 256, 0, st, d_ctx, p->use_pdl && !p->timeline);
        n_kernels += 2;
        mark(st, "k_cost_eval", true);
        if (R > 1)
          launch_after(k_cost_eval<4>, dim3(gxc, R), warps_c * 32, smem_c, st, d_ctx, p->use_pdl && !p->timeline);
        else
          launch_after(k_cost_eval<1>, dim3(gxc, R), warps_c * 32, smem_c, st, d_ctx, p->use_pdl && !p->timeline);
      } else {
        mark(st, "k_cost_eval", true);
        if (R > 1)
          k_cost_eval<4><<<dim3(gxc, R), warps_c * 32, smem_c, st>>>(d_ctx);
        else
          k_cost_eval<1><<<dim3(gxc, R), warps_c * 32, smem_c, st>>>(d_ctx);
      }
      mark(st, "k_cost_eval", false);
      n_kernels += 1;
    }
    if (eval_stop) KC_CUDA(cudaEventRecord(eval_stop, st));
  }
  return KC_OK;
}

// One cycle = memset(s) + up to twelve kernels whose only argument is the ctx pointer (k_scatter also takes
// the number of its classifying CTAs, a function of the launch geometry), so the launch
// set is captured once per launch geometry into a CUDA graph and replayed with a single call (the
// per-cycle inputs travel through the ctx / staging buffers, not through kernel arguments).
int32_t launch_cycle(kc_planner *p, const RobotCtx *d_ctx, int R, size_t zero_words_total,
                     size_t sph_words_total, int32_t max_sensor, int32_t max_slots, int P, int S,
                     bool any_points, int mode /*0 cycle, 1 sampler*/, cudaEvent_t eval_start,
                     cudaEvent_t eval_stop, int32_t max_qcells, int32_t dil_words) {
  if (max_slots > 0) {  // function attributes are not stream work: set them outside any capture
    size_t smem_r = 0, smem_c = 0;
    pick_rollout_warps(P, dil_words, smem_r);
    pick_cost_warps(P, S, smem_c);
    if (mode == 0) {
      KC_TRY(allow_smem(k_rollout_collide<false, false>, smem_r));
      if (p->general_bound) KC_TRY(allow_smem(k_rollout_collide<false, true>, smem_r));
      KC_TRY(allow_smem(k_cost_eval<1>, smem_c));
      KC_TRY(allow_smem(k_cost_eval<4>, smem_c));
      KC_TRY(allow_smem(k_cost_bounds, smem_c));
      const int wc = pick_cost_warps(P, S, smem_c);
      if (R > 1)
        KC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&p->cost_ctas_per_sm, k_cost_eval<4>, wc * 32, smem_c));
      else
        KC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&p->cost_ctas_per_sm, k_cost_eval<1>, wc * 32, smem_c));
      KC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&p->bounds_ctas_per_sm, k_cost_bounds, wc * 32, smem_c));
    } else {
      KC_TRY(allow_smem(k_rollout_collide<true, false>, smem_r));
      if (p->general_bound) KC_TRY(allow_smem(k_rollout_collide<true, true>, smem_r));
    }
  }
  int n_kernels = 0;
  if (eval_start || eval_stop || !p->use_graphs || R > 1 || p->timeline) {  // a batch chunk is milliseconds of work
    KC_TRY(enqueue_cycle(p, d_ctx, R, zero_words_total, sph_words_total, max_sensor, max_slots, P, S,
                         any_points, mode, eval_start, eval_stop, max_qcells, dil_words, n_kernels));
    p->launches += n_kernels;
    KC_CUDA(cudaGetLastError());
    return KC_OK;
  }
  const kc_planner::GraphKey key{d_ctx, p->d_zero.ptr, p->d_sph.ptr, zero_words_total, sph_words_total,
                                 R, max_sensor, max_slots, P, S, mode, max_qcells, dil_words, any_points,
                                 p->heavy_bound, p->general_bound};
  kc_planner::GraphSlot *slot = nullptr, *victim = &p->graphs[0];
  for (kc_planner::GraphSlot &g : p->graphs) {
    if (g.exec && g.key == key) slot = &g;
    if (g.stamp < victim->stamp) victim = &g;
  }
  if (!slot) {
    slot = victim;  // least recently used
    if (slot->exec) {
      cudaGraphExecDestroy(slot->exec);
      slot->exec = nullptr;
    }
    cudaGraph_t graph = nullptr;
    KC_CUDA(cudaStreamBeginCapture(p->stream, cudaStreamCaptureModeThreadLocal));
    const int32_t rc = enqueue_cycle(p, d_ctx, R, zero_words_total, sph_words_total, max_sensor,
                                     max_slots, P, S, any_points, mode, nullptr, nullptr, max_qcells,
                                     dil_words, n_kernels);
    const cudaError_t e = cudaStreamEndCapture(p->stream, &graph);
    if (rc != KC_OK) {
      if (graph) cudaGraphDestroy(graph);
      return rc;
    }
    KC_CUDA(e);
    const cudaError_t ei = cudaGraphInstantiate(&slot->exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ei != cudaSuccess) slot->exec = nullptr;
    KC_CUDA(ei);
    slot->key = key;
    slot->kernels = n_kernels;
  }
  slot->stamp = ++p->graph_clock;
  KC_CUDA(cudaGraphLaunch(slot->exec, p->stream));
  p->launches += slot->kernels;
  return KC_OK;
}

void fill_result(kc_planner *p, const uint8_t *host_res, int P, int n_slots, kc_cycle_result *out) {
  const ResultHeader *h = reinterpret_cast<const ResultHeader *>(host_res);
  const float *rows = reinterpret_cast<const float *>(host_res + sizeof(ResultHeader));
  out->found = h->found;
  out->cost = h->cost;
  out->slot = h->slot;
  out->n_points = P;
  out->n_slots = n_slots;
  out->n_admissible = h->n_admissible;
  if (h->n_admissible == 0) {  // ref: dwa.h:219-221 -> {Trajectory2D(), false, 0.0}
    out->found = 0;
    out->cost = 0.0f;
  }
  out->vx = rows;
  out->vy = rows + (P - 1);
  out->omega = rows + 2 * (P - 1);
  out->x = rows + 3 * (P - 1);
  out->y = rows + 3 * (P - 1) + P;
  p->heavy_seen = h->heavy_cells != 0;  // feedback for the next cycle's launch set (heavy_kernel_on)
}

// stage [ctx | axes | sensor] for one robot into the pinned buffer; returns layout offsets
struct StageLayout {
  size_t ctx_off, vx_off, vy_off, om_off, row_off, sensor_off, total;
};
StageLayout plan_stage(const Axes &ax, const SensorDesc &sd) {
  StageLayout L;
  size_t o = 0;
  L.ctx_off = o;
  o = align_up(o + sizeof(RobotCtx));
  L.vx_off = o;
  o += ax.vx.size() * 8;
  L.vy_off = o;
  o += ax.vy.size() * 8;
  L.om_off = o;
  o += ax.om.size() * 8;
  L.row_off = o;
  o = align_up(o + ax.row_off.size() * 4);
  L.sensor_off = o;
  if (!sd.dev) o += sd.is_cloud ? (size_t)sd.n * 12 : (size_t)sd.n * 16;
  L.total = align_up(o);
  return L;
}

// developer: KOMPASS_B200_HOST_PROF=1 prints the mean host-side phase times of run_single to stderr
struct HostProf {
  bool on = getenv("KOMPASS_B200_HOST_PROF") != nullptr;
  double acc[8] = {0};
  long n = 0;
  std::chrono::steady_clock::time_point t;
  void start() { if (on) t = std::chrono::steady_clock::now(); }
  void lap(int i) {
    if (!on) return;
    const auto now = std::chrono::steady_clock::now();
    acc[i] += std::chrono::duration<double, std::micro>(now - t).count();
    t = now;
  }
  ~HostProf() {
    if (on && n)
      fprintf(stderr, "[kompass_b200 host prof] %ld cycles, mean us: prepare %.2f | stage+H2D enqueue %.2f | launch %.2f | "
              "wait for the record %.2f | fill result %.2f\n", n, acc[0] / n, acc[1] / n, acc[2] / n, acc[3] / n, acc[4] / n);
  }
};
static HostProf g_host_prof;

int32_t run_single(kc_planner *p, const double vel[3], const double pose[3], const SensorDesc &sd,
                   int32_t seg_start, int32_t seg_count, int mode, kc_cycle_result *out) {
  KC_REQUIRE(p && vel && pose, KC_ERR_INVALID_ARG, "null argument");
  g_host_prof.start();
  KC_REQUIRE(sd.n >= 0, KC_ERR_INVALID_ARG, "negative point count");
  if (mode == 0)
    KC_REQUIRE(p->path_n >= 2, KC_ERR_INVALID_ARG,
               "Pointer to global path is NULL. Cannot use DWA local planner without setting a "
               "global path");
  p->heavy_bound = p->heavy_kernel_on();
  Axes ax;
  enumerate_axes(p->cfg, vel, ax);
  RobotCtx cx;
  Sizes sz;
  const float D = p->cfg.max_local_range / 3.0f;  // ref: cost_evaluator.h:179 via dwa.h:223
  p->general_bound = false;
  KC_TRY(fill_ctx_scalars(p, p->P, own_path(p), vel, pose, sd, seg_start, seg_count, true, mode == 0, D, pose,
                          ax, cx, sz));
  p->general_bound = cx.coll_general != 0;  // tilted mount + scan: the oriented-cube rollout kernel
  const double reach = ax.max_speed * (double)(p->P - 1) * cx.dt * 1.001 + 1e-3;
  set_grid_window(cx, (float)pose[0], (float)pose[1], reach + (double)D * 1.001 + 1e-3, reach + 1e-3);

  const size_t zw = zero_words_per_robot(sz.bitmap_words);
  KC_TRY(reserve_workspace(p, 1, zw, sz.sph_words, sd.n, ax.n_slots, p->P));
  bind_workspace(p, cx, own_path(p), 0, zw, sz.bitmap_words, sz.sph_words, sd.n, ax.n_slots, p->P);
  const int32_t dil_words = plan_dilation(cx, sz.bitmap_words);
  if (mode == 1) {
    const size_t nv = (size_t)ax.n_slots * (p->P - 1);
    KC_TRY(p->d_rows.reserve(3 * nv + 16));
    cx.rows_vx = p->d_rows.ptr;
    cx.rows_vy = cx.rows_vx + nv;
    cx.rows_om = cx.rows_vy + nv;
  }

  g_host_prof.lap(0);
  const StageLayout L = plan_stage(ax, sd);
  KC_TRY(p->h_stage.reserve(L.total));
  KC_TRY(p->d_stage.reserve(L.total));
  uint8_t *hs = p->h_stage.ptr;
  uint8_t *ds = p->d_stage.ptr;
  cx.ax_vx = reinterpret_cast<const double *>(ds + L.vx_off);
  cx.ax_vy = reinterpret_cast<const double *>(ds + L.vy_off);
  cx.ax_om = reinterpret_cast<const double *>(ds + L.om_off);
  cx.row_off = reinterpret_cast<const int32_t *>(ds + L.row_off);
  cx.sensor = sd.dev ? sd.dev : (ds + L.sensor_off);
  // caller buffers that are already page-locked (kc_pinned_alloc, cudaHostAlloc, cudaHostRegister)
  // are read by the DMA engine directly: no staging copy
  auto pinned = [](const void *q) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, q) != cudaSuccess) {
      cudaGetLastError();
      return false;
    }
    return a.type == cudaMemoryTypeHost;
  };
  const bool src_pinned = !sd.dev && sd.n > 0 && pinned(sd.host) && (sd.is_cloud || pinned(sd.host2));
  bool in_place = false;
  if (src_pinned && sd.is_cloud && p->zero_copy_cloud) {
    // the only reader of the raw cloud is k_prep_points (one coalesced pass): let it pull the points
    // over PCIe itself instead of waiting for a DMA into HBM first
    void *dp = nullptr;
    if (cudaHostGetDevicePointer(&dp, const_cast<void *>(sd.host), 0) == cudaSuccess && dp) {
      cx.sensor = dp;
      in_place = true;
    } else {
      cudaGetLastError();
    }
  }
  // a pageable cloud goes through the page-locked staging buffer (copy pool, kc_hostcopy.h) and is
  // then read in place the same way
  bool staged_in_place = false;
  if (!src_pinned && !sd.dev && sd.n > 0 && sd.is_cloud && p->zero_copy_cloud) {
    void *dp = nullptr;
    if (cudaHostGetDevicePointer(&dp, hs + L.sensor_off, 0) == cudaSuccess && dp) {
      cx.sensor = dp;
      in_place = staged_in_place = true;
    } else {
      cudaGetLastError();
    }
  }
  bool result_in_host = false;
  if (mode == 0 && p->mapped_result && ax.n_slots > 0) {
    void *dp = nullptr;
    if (cudaHostGetDevicePointer(&dp, p->h_result.ptr, 0) == cudaSuccess && dp) {
      cx.result = reinterpret_cast<ResultHeader *>(dp);
      cx.res_rows = reinterpret_cast<float *>(reinterpret_cast<uint8_t *>(dp) + sizeof(ResultHeader));
      result_in_host = true;
      if (++p->cycle_seq == 0) p->cycle_seq = 1;
      cx.seq = p->cycle_seq;
      reinterpret_cast<volatile ResultHeader *>(p->h_result.ptr)->seq = 0;
    } else {
      cudaGetLastError();
    }
  }
  memcpy(hs + L.ctx_off, &cx, sizeof(cx));
  if (!ax.vx.empty()) memcpy(hs + L.vx_off, ax.vx.data(), ax.vx.size() * 8);
  if (!ax.vy.empty()) memcpy(hs + L.vy_off, ax.vy.data(), ax.vy.size() * 8);
  if (!ax.om.empty()) memcpy(hs + L.om_off, ax.om.data(), ax.om.size() * 8);
  memcpy(hs + L.row_off, ax.row_off.data(), ax.row_off.size() * 4);
  // header (ctx + axes) first, then the sensor data in chunks: the copy of chunk k+1 into pinned
  // memory overlaps the DMA of chunk k. Invariant that keeps the staging buffer (and a caller cloud
  // read in place) free for the next cycle even when the previous one returned on the polled result
  // record without a stream sync: every H2D copy and every kernel that reads h_stage / the caller's
  // cloud precedes, in stream order, the kernel that publishes the record - nothing may read them
  // after the publish.
  KC_CUDA(cudaMemcpyAsync(ds, hs, std::min(L.sensor_off, L.total), cudaMemcpyHostToDevice, p->stream));
  if (staged_in_place)
    CopyPool::instance().copy(hs + L.sensor_off, static_cast<const uint8_t *>(sd.host), (size_t)sd.n * 12,
                              CopyPool::piece_for((size_t)sd.n * 12), [](size_t, size_t) {}, (size_t)sd.n * 12);
  if (!sd.dev && sd.n > 0 && !in_place) {
    const size_t half = (size_t)sd.n * 8;
    const size_t bytes = sd.is_cloud ? (size_t)sd.n * 12 : 2 * half;
    constexpr size_t kChunk = 192 * 1024;
    if (src_pinned) {
      if (sd.is_cloud) {
        KC_CUDA(cudaMemcpyAsync(ds + L.sensor_off, sd.host, bytes, cudaMemcpyHostToDevice, p->stream));
      } else {
        KC_CUDA(cudaMemcpyAsync(ds + L.sensor_off, sd.host, half, cudaMemcpyHostToDevice, p->stream));
        KC_CUDA(cudaMemcpyAsync(ds + L.sensor_off + half, sd.host2, half, cudaMemcpyHostToDevice, p->stream));
      }
    } else if (sd.is_cloud) {
      // pageable cloud: the copy pool's threads and this one copy pieces into the page-locked staging
      // buffer, finished runs go to the DMA engine in order (kc_hostcopy.h)
      cudaError_t err = cudaSuccess;
      CopyPool::instance().copy(hs + L.sensor_off, static_cast<const uint8_t *>(sd.host), bytes,
                                CopyPool::piece_for(bytes), [&](size_t off, size_t len) {
                                  if (err == cudaSuccess)
                                    err = cudaMemcpyAsync(ds + L.sensor_off + off, hs + L.sensor_off + off, len,
                                                          cudaMemcpyHostToDevice, p->stream);
                                }, bytes / 3);
      KC_CUDA(err);
    } else
    for (size_t off = 0; off < bytes; off += kChunk) {
      const size_t len = std::min(kChunk, bytes - off);
      if (sd.is_cloud) {
        memcpy(hs + L.sensor_off + off, (const uint8_t *)sd.host + off, len);
      } else {  // ranges then angles, from two caller arrays
        const size_t a0 = off, a1 = off + len;
        if (a0 < half)
          memcpy(hs + L.sensor_off + a0, (const uint8_t *)sd.host + a0, std::min(a1, half) - a0);
        if (a1 > half) {
          const size_t b0 = std::max(a0, half);
          memcpy(hs + L.sensor_off + b0, (const uint8_t *)sd.host2 + (b0 - half), a1 - b0);
        }
      }
      KC_CUDA(cudaMemcpyAsync(ds + L.sensor_off + off, hs + L.sensor_off + off, len,
                              cudaMemcpyHostToDevice, p->stream));
    }
  }
  const RobotCtx *d_ctx = reinterpret_cast<const RobotCtx *>(ds + L.ctx_off);
  g_host_prof.lap(1);
  KC_TRY(launch_cycle(p, d_ctx, 1, zw, sz.sph_words, sd.n, ax.n_slots, p->P, cx.seg_count,
                      sd.n > 0, mode, nullptr, nullptr, qcells(cx), dil_words));
  g_host_prof.lap(2);
  p->last_slots = ax.n_slots;
  p->last_was_cycle = (mode == 0);
  p->last_replay = false;
  p->last_ctx = cx;
  if (mode == 0) {
    const size_t res_bytes = sizeof(ResultHeader) + sizeof(float) * 5 * (size_t)p->P;
    if (ax.n_slots > 0) {
      if (!result_in_host)
        KC_CUDA(cudaMemcpyAsync(p->h_result.ptr, p->d_result.ptr, res_bytes, cudaMemcpyDeviceToHost,
                                p->stream));
      if (result_in_host && p->poll_result) {
        // the winner record lands in mapped pinned memory, its sequence number last: watch for it
        // instead of paying the driver's completion latency (the stream is checked now and then so
        // that a failed launch still surfaces as an error)
        volatile ResultHeader *hr = reinterpret_cast<volatile ResultHeader *>(p->h_result.ptr);
        for (unsigned spins = 0; hr->seq != cx.seq; ++spins) {
          if ((spins & 0x3fff) == 0x3fff) {
            const cudaError_t q = cudaStreamQuery(p->stream);
            if (q == cudaSuccess) break;  // finished (no slot survived to publish: cannot happen, but stay safe)
            if (q != cudaErrorNotReady) KC_CUDA(q);
          }
#if defined(__x86_64__)
          __builtin_ia32_pause();
#endif
        }
        if (hr->seq != cx.seq) KC_CUDA(cudaStreamSynchronize(p->stream));
        // acquire: the row loads of fill_result must not be hoisted above the sequence-number load
        // (they cannot on x86; an aarch64 host such as Grace may reorder them)
        std::atomic_thread_fence(std::memory_order_acquire);
      } else {
        KC_CUDA(cudaStreamSynchronize(p->stream));
      }
    } else {
      memset(p->h_result.ptr, 0, res_bytes);
    }
    g_host_prof.lap(3);
    if (out) fill_result(p, p->h_result.ptr, p->P, ax.n_slots, out);
    g_host_prof.lap(4);
    g_host_prof.n += 1;
  }
  return KC_OK;
}

bool host_page_locked(const void *q) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, q) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost;
}

// Host -> device upload of several large arrays that live in ordinary pageable memory (the sample
// batches of CostEvaluator::getMinTrajectoryCost: 100 MB at the reference's benchmark shape). A
// pageable cudaMemcpy is staged by the driver on one thread at ~10 GB/s; here the process's copy pool
// (kc_hostcopy.h) and this thread copy 1 MB pieces into the handle's page-locked staging buffer and
// every finished run of pieces goes to the DMA engine in order, so the copy into page-locked memory
// runs at several cores' memory bandwidth and overlaps the PCIe transfer. Page-locked sources are
// DMA-ed directly.
struct UploadPart {
  void *dst;
  const void *src;
  size_t bytes;
};
int32_t upload_pageable(kc_planner *p, const std::vector<UploadPart> &parts, cudaStream_t st) {
  size_t total = 0;
  bool all_pinned = true;
  for (const UploadPart &u : parts) {
    total += u.bytes;
    if (u.bytes && !host_page_locked(u.src)) all_pinned = false;
  }
  constexpr size_t kPiece = 1 << 20;
  if (all_pinned || total < 8 * kPiece) {  // small or already page-locked: plain copies
    for (const UploadPart &u : parts)
      if (u.bytes) KC_CUDA(cudaMemcpyAsync(u.dst, u.src, u.bytes, cudaMemcpyHostToDevice, st));
    return KC_OK;
  }
  // the staging buffer is reused by the next call: everything queued from it must have left first
  KC_CUDA(cudaStreamSynchronize(st));
  KC_TRY(p->h_bulk.reserve(total));
  uint8_t *stage = p->h_bulk.ptr;
  cudaError_t err = cudaSuccess;
  size_t base = 0;
  for (const UploadPart &u : parts) {
    if (!u.bytes) continue;
    uint8_t *dst = static_cast<uint8_t *>(u.dst);
    CopyPool::instance().copy(stage + base, static_cast<const uint8_t *>(u.src), u.bytes, kPiece,
                              [&](size_t off, size_t len) {
                                if (err == cudaSuccess)
                                  err = cudaMemcpyAsync(dst + off, stage + base + off, len, cudaMemcpyHostToDevice, st);
                              });
    base += u.bytes;
  }
  KC_CUDA(err);
  return KC_OK;
}

int32_t run_sampler(kc_planner *p, const double vel[3], const double pose[3], const SensorDesc &sd,
                    kc_samples *out) {
  KC_REQUIRE(out, KC_ERR_INVALID_ARG, "null output");
  KC_TRY(run_single(p, vel, pose, sd, 0, 0, 1, nullptr));
  const int n = p->last_slots, P = p->P;
  memset(out, 0, sizeof(*out));
  out->n_points = P;
  if (n == 0) return KC_OK;
  const size_t nv = (size_t)n * (P - 1), np = (size_t)n * P;
  KC_TRY(p->d_dst.reserve((size_t)n + 1));
  KC_TRY(p->d_crows.reserve(3 * nv + 2 * np + 16));
  KC_TRY(p->d_cslots.reserve(n));
  int32_t *d_count = p->d_dst.ptr + n;
  k_compact_index<<<1, 1024, 0, p->stream>>>(p->d_adm.ptr, n, p->d_dst.ptr, d_count);
  float *cvx = p->d_crows.ptr, *cvy = cvx + nv, *com = cvy + nv, *cxx = com + nv, *cyy = cxx + np;
  const RobotCtx *d_ctx = reinterpret_cast<const RobotCtx *>(p->d_stage.ptr);
  k_compact_rows<<<n, 64, 0, p->stream>>>(d_ctx, p->d_dst.ptr, cvx, cvy, com, cxx, cyy,
                                          p->d_cslots.ptr);
  p->launches += 2;
  KC_CUDA(cudaGetLastError());
  int32_t count = 0;
  KC_CUDA(cudaMemcpyAsync(&count, d_count, 4, cudaMemcpyDeviceToHost, p->stream));
  KC_CUDA(cudaStreamSynchronize(p->stream));
  const size_t cv = (size_t)count * (P - 1), cp = (size_t)count * P;
  const size_t bytes = (3 * cv + 2 * cp) * 4 + (size_t)count * 4;
  KC_TRY(p->h_samples.reserve(bytes + 64));
  float *h = reinterpret_cast<float *>(p->h_samples.ptr);
  if (count > 0) {
    KC_CUDA(cudaMemcpyAsync(h, cvx, cv * 4, cudaMemcpyDeviceToHost, p->stream));
    KC_CUDA(cudaMemcpyAsync(h + cv, cvy, cv * 4, cudaMemcpyDeviceToHost, p->stream));
    KC_CUDA(cudaMemcpyAsync(h + 2 * cv, com, cv * 4, cudaMemcpyDeviceToHost, p->stream));
    KC_CUDA(cudaMemcpyAsync(h + 3 * cv, cxx, cp * 4, cudaMemcpyDeviceToHost, p->stream));
    KC_CUDA(cudaMemcpyAsync(h + 3 * cv + cp, cyy, cp * 4, cudaMemcpyDeviceToHost, p->stream));
    KC_CUDA(cudaMemcpyAsync(h + 3 * cv + 2 * cp, p->d_cslots.ptr, (size_t)count * 4,
                            cudaMemcpyDeviceToHost, p->stream));
    KC_CUDA(cudaStreamSynchronize(p->stream));
  }
  out->count = count;
  out->vx = h;
  out->vy = h + cv;
  out->omega = h + 2 * cv;
  out->x = h + 3 * cv;
  out->y = h + 3 * cv + cp;
  out->slots = reinterpret_cast<const int32_t *>(h + 3 * cv + 2 * cp);
  return KC_OK;
}

int32_t validate_config(const kc_planner_config *c) {
  KC_REQUIRE(c, KC_ERR_INVALID_ARG, "null config");
  KC_REQUIRE(c->control_type >= 0 && c->control_type <= 2, KC_ERR_INVALID_ARG, "Invalid control type");
  KC_REQUIRE(c->robot_shape >= 0 && c->robot_shape <= 2, KC_ERR_INVALID_ARG,
             "Invalid robot geometry type");
  // parameter ranges of the reference Parameter classes (trajectory_sampler.h:24-58)
  KC_REQUIRE(c->time_step >= 0.001 && c->time_step <= 1000.0, KC_ERR_OUT_OF_RANGE,
             "time_step out of range [0.001, 1000]");
  KC_REQUIRE(c->prediction_horizon >= 0.001 && c->prediction_horizon <= 1000.0, KC_ERR_OUT_OF_RANGE,
             "prediction_horizon out of range [0.001, 1000]");
  KC_REQUIRE(c->control_horizon >= 0.001 && c->control_horizon <= 1000.0, KC_ERR_OUT_OF_RANGE,
             "control_horizon out of range [0.001, 1000]");
  KC_REQUIRE(c->max_linear_samples >= 1 && c->max_linear_samples <= 1000, KC_ERR_OUT_OF_RANGE,
             "max_linear_samples out of range [1, 1000]");
  KC_REQUIRE(c->max_angular_samples >= 1 && c->max_angular_samples <= 1000, KC_ERR_OUT_OF_RANGE,
             "max_angular_samples out of range [1, 1000]");
  KC_REQUIRE(c->octree_resolution > 0.0 && c->octree_resolution <= 1000.0, KC_ERR_OUT_OF_RANGE,
             "octree_map_resolution out of range (0, 1000]");
  const double ws[5] = {c->w_path, c->w_goal, c->w_obstacles, c->w_smooth, c->w_jerk};
  for (double w : ws)
    KC_REQUIRE(w >= 0.0 && w <= 1000.0, KC_ERR_OUT_OF_RANGE, "cost weight out of range [0, 1000]");
  return KC_OK;
}

}  // namespace

// =================================================================================================
// C-ABI
// =================================================================================================
extern "C" {

int32_t kc_planner_create(const kc_planner_config *cfg, kc_planner **out) {
  KC_REQUIRE(out, KC_ERR_INVALID_ARG, "null output handle");
  *out = nullptr;
  KC_TRY(validate_config(cfg));
  KC_TRY(ensure_device());
  kc_planner *p = new kc_planner();
  p->cfg = *cfg;
  if (p->cfg.num_ctrl_points < 0)
    p->cfg.num_ctrl_points = (int64_t)(size_t)(cfg->control_horizon / cfg->time_step);
  if (p->cfg.max_local_range <= 0.0f) p->cfg.max_local_range = 10.0f;
  p->base_horizon = p->horizon = cfg->prediction_horizon;
  p->P = (int32_t)(size_t)(cfg->prediction_horizon / cfg->time_step);  // trajectory.h:48-51
  if (p->P < 2) {
    delete p;
    set_error("prediction_horizon / time_step must give at least 2 points per trajectory");
    return KC_ERR_INVALID_ARG;
  }
  p->sensor_tf_body = hm::rigid_from_quat(cfg->sensor_rotation, cfg->sensor_position);
  // the main chain (grid preparation -> candidate lists -> cost kernel) is the critical path: its
  // CTAs are scheduled ahead of the two side branches, which have slack (KC_STREAM_PRIO=0 disables)
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
  const char *pd = getenv("KC_PDL");  // KC_PDL=0: plain stream-ordered launches everywhere
  p->use_pdl = !(pd && pd[0] == '0');
  const char *pe = getenv("KC_STREAM_PRIO");
  if (pe && pe[0] == '0') prio_hi = prio_lo = 0;
  cudaError_t e = cudaStreamCreateWithPriority(&p->stream, cudaStreamNonBlocking, prio_hi);
  if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&p->side, cudaStreamNonBlocking, prio_lo);
  if (e == cudaSuccess) e = cudaEventCreate(&p->ev0);
  if (e == cudaSuccess) e = cudaEventCreate(&p->ev1);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->ev_join, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&p->side2, cudaStreamNonBlocking, prio_lo);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->ev_fork2, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->ev_join2, cudaEventDisableTiming);
  if (e != cudaSuccess) {
    delete p;
    return cuda_fail(e, "stream/event creation", __FILE__, __LINE__);
  }
  *out = p;
  return KC_OK;
}

void kc_planner_destroy(kc_planner *p) {
  kc::ensure_device();  // the handle's device on this thread (frees below)
  if (!p) return;
  if (p->stream) cudaStreamSynchronize(p->stream);
  p->d_path.release();
  p->h_stage.release();
  p->d_stage.release();
  p->h_bulk.release();
  p->d_zero.release();
  p->d_dil.release();
  p->d_sph.release();
  p->d_tab_sc.release();
  p->d_tab_yaw.release();
  p->d_bf_xy.release();
  p->d_bf_min.release();
  p->d_bf_cost.release();
  p->d_cell_start.release();
  p->d_cell_cursor.release();
  p->d_work_cells.release();
  p->d_pwork_cells.release();
  p->d_cell_nn.release();
  p->d_row_dx.release();
  p->d_cell_info.release();
  p->d_cand.release();
  p->d_pcell_info.release();
  p->d_pcand.release();
  p->d_list.release();
  p->d_cutv.release();
  p->d_rowsxy.release();
  p->d_tmp_cell.release();
  p->d_tmp_xy.release();
  p->d_sorted_xy.release();
  p->d_costs.release();
  p->d_adm.release();
  p->d_prn.release();
  p->d_lbv.release();
  p->d_ubd.release();
  p->d_sjv.release();
  p->d_surv.release();
  p->d_dmin.release();
  p->d_dbg.release();
  p->d_result.release();
  p->h_result.release();
  p->d_rows.release();
  p->d_crows.release();
  p->d_dst.release();
  p->d_cslots.release();
  p->h_samples.release();
  p->d_in.release();
  p->d_bbox.release();
  p->h_costs.release();
  p->h_adm.release();
  p->d_bank.release();
  p->d_batch_xyz.release();
  p->d_batch_scan.release();
  p->h_batch_scan.release();
  p->d_batch_stage.release();
  for (kc_planner::GraphSlot &g : p->graphs)
    if (g.exec) cudaGraphExecDestroy(g.exec);
  for (cudaEvent_t e : p->evk) cudaEventDestroy(e);
  if (p->ev0) cudaEventDestroy(p->ev0);
  if (p->ev1) cudaEventDestroy(p->ev1);
  for (cudaEvent_t e : p->tl_ev)
    if (e) cudaEventDestroy(e);
  if (p->ev_fork) cudaEventDestroy(p->ev_fork);
  if (p->ev_join) cudaEventDestroy(p->ev_join);
  if (p->ev_fork2) cudaEventDestroy(p->ev_fork2);
  if (p->ev_join2) cudaEventDestroy(p->ev_join2);
  if (p->side2) cudaStreamDestroy(p->side2);
  if (p->copy) cudaStreamDestroy(p->copy);
  if (p->ev_copy) cudaEventDestroy(p->ev_copy);
  if (p->side) cudaStreamDestroy(p->side);
  if (p->stream) cudaStreamDestroy(p->stream);
  delete p;
}

int32_t kc_planner_set_weights(kc_planner *p, double w_path, double w_goal, double w_obstacles,
                               double w_smooth, double w_jerk) {
  KC_REQUIRE(p, KC_ERR_INVALID_ARG, "null handle");
  KC_TRY(kc::ensure_device());
  const double ws[5] = {w_path, w_goal, w_obstacles, w_smooth, w_jerk};
  for (double w : ws)
    KC_REQUIRE(w >= 0.0 && w <= 1000.0, KC_ERR_OUT_OF_RANGE, "cost weight out of range [0, 1000]");
  p->cfg.w_path = w_path;
  p->cfg.w_goal = w_goal;
  p->cfg.w_obstacles = w_obstacles;
  p->cfg.w_smooth = w_smooth;
  p->cfg.w_jerk = w_jerk;
  return KC_OK;
}

int32_t kc_planner_set_octree_resolution(kc_planner *p, double resolution) {
  KC_REQUIRE(p, KC_ERR_INVALID_ARG, "null handle");
  KC_REQUIRE(resolution > 0.0, KC_ERR_OUT_OF_RANGE, "octree resolution must be positive");
  KC_TRY(kc::ensure_device());
  p->cfg.octree_resolution = resolution;
  return KC_OK;
}

int32_t kc_planner_set_drop_samples(kc_planner *p, int32_t drop) {
  KC_REQUIRE(p, KC_ERR_INVALID_ARG, "null handle");
  KC_TRY(kc::ensure_device());
  p->cfg.drop_samples = drop ? 1 : 0;
  return KC_OK;
}

int32_t kc_planner_set_max_range(kc_planner *p, float max_range) {
  KC_REQUIRE(p, KC_ERR_INVALID_ARG, "null handle");
  KC_REQUIRE(max_range > 0.0f, KC_ERR_OUT_OF_RANGE, "max range must be positive");
  KC_TRY(kc::ensure_device());
  p->cfg.max_local_range = max_range;
  return KC_OK;
}

float kc_planner_get_max_range(const kc_planner *p) { return p ? p->cfg.max_local_range : 0.0f; }
int32_t kc_planner_num_slots_last(const kc_planner *p) { return p ? p->last_slots : 0; }

int32_t kc_planner_set_prediction_horizon(kc_planner *p, double horizon, int32_t *n_points) {
  KC_REQUIRE(p, KC_ERR_INVALID_ARG, "null handle");
  KC_TRY(kc::ensure_device());
  p->P = horizon_points(p->cfg.time_step, p->base_horizon, horizon);
  p->horizon = horizon;
  if (n_points) *n_points = p->P;
  return KC_OK;
}

int32_t kc_planner_num_trajectories(const kc_planner *p) {
  if (!p) return 0;
  int nx, ny;
  linear_split(p->cfg.control_type, p->cfg.max_linear_samples, nx, ny);
  const int nang = p->cfg.max_angular_samples + 1 - (p->cfg.max_angular_samples % 2);
  return p->cfg.control_type == KC_OMNI ? nx * nang + nx * ny : nx * nang;
}

int32_t kc_planner_num_points(const kc_planner *p) { return p ? p->P : 0; }

int32_t kc_planner_set_path(kc_planner *p, const float *X, const float *Y, const float *acc,
                            int32_t n, float total_length) {
  KC_REQUIRE(p && X && Y && acc, KC_ERR_INVALID_ARG, "null argument");
  KC_REQUIRE(n >= 2, KC_ERR_INVALID_ARG, "At least two points are required to create a path.");
  KC_TRY(kc::ensure_device());
  KC_TRY(p->d_path.reserve(3 * (size_t)n));
  KC_CUDA(cudaStreamSynchronize(p->stream));
  KC_CUDA(cudaMemcpy(p->d_path.ptr, X, (size_t)n * 4, cudaMemcpyHostToDevice));
  KC_CUDA(cudaMemcpy(p->d_path.ptr + n, Y, (size_t)n * 4, cudaMemcpyHostToDevice));
  KC_CUDA(cudaMemcpy(p->d_path.ptr + 2 * (size_t)n, acc, (size_t)n * 4, cudaMemcpyHostToDevice));
  p->hX.assign(X, X + n);
  p->hY.assign(Y, Y + n);
  p->path_n = n;
  p->path_len = total_length;
  return KC_OK;
}

int32_t kc_planner_cycle_scan(kc_planner *p, const double vel[3], const double pose[3],
                              const double *ranges, const double *angles, int32_t n,
                              int32_t seg_start, int32_t seg_count, kc_cycle_result *out) {
  KC_REQUIRE(p && out, KC_ERR_INVALID_ARG, "null argument");
  KC_REQUIRE(n == 0 || (ranges && angles), KC_ERR_INVALID_ARG, "null scan arrays");
  KC_TRY(kc::ensure_device());
  SensorDesc sd;
  sd.is_cloud = 0;
  sd.n = n;
  sd.host = ranges;
  sd.host2 = angles;
  return run_single(p, vel, pose, sd, seg_start, seg_count, 0, out);
}

int32_t kc_planner_cycle_cloud(kc_planner *p, const double vel[3], const double pose[3],
                               const float *xyz, int32_t n, int32_t seg_start, int32_t seg_count,
                               kc_cycle_result *out) {
  KC_REQUIRE(p && out, KC_ERR_INVALID_ARG, "null argument");
  KC_REQUIRE(n == 0 || xyz, KC_ERR_INVALID_ARG, "null cloud");
  KC_TRY(kc::ensure_device());
  SensorDesc sd;
  sd.is_cloud = 1;
  sd.n = n;
  sd.host = xyz;
  return run_single(p, vel, pose, sd, seg_start, seg_count, 0, out);
}

int32_t kc_planner_fetch_costs(kc_planner *p, float *costs, uint8_t *admissible) {
  KC_REQUIRE(p, KC_ERR_INVALID_ARG, "null handle");
  KC_TRY(kc::ensure_device());
  const int n = p->last_slots;
  if (n <= 0) return KC_OK;
  KC_CUDA(cudaStreamSynchronize(p->stream));
  if (costs) KC_CUDA(cudaMemcpy(costs, p->d_costs.ptr, (size_t)n * 4, cudaMemcpyDeviceToHost));
  if (admissible) KC_CUDA(cudaMemcpy(admissible, p->d_adm.ptr, (size_t)n, cudaMemcpyDeviceToHost));
  return KC_OK;
}

// 1 where the cost reported by kc_planner_fetch_costs is only a lower bound of the slot's total: the
// branch and bound proved that the slot cannot win and skipped its exact obstacle search
int32_t kc_planner_fetch_pruned(kc_planner *p, uint8_t *pruned) {
  KC_REQUIRE(p && pruned, KC_ERR_INVALID_ARG, "null argument");
  KC_TRY(kc::ensure_device());
  const int n = p->last_slots;
  if (n <= 0) return KC_OK;
  KC_CUDA(cudaStreamSynchronize(p->stream));
  if (!p->prune_for(n) || !p->last_was_cycle) {
    memset(pruned, 0, (size_t)n);
    return KC_OK;
  }
  KC_CUDA(cudaMemcpy(pruned, p->d_prn.ptr, (size_t)n, cudaMemcpyDeviceToHost));
  // slots that are not admissible never reach the cost kernels: their flag bytes are stale
  std::vector<uint8_t> adm((size_t)n);
  KC_CUDA(cudaMemcpy(adm.data(), p->d_adm.ptr, (size_t)n, cudaMemcpyDeviceToHost));
  for (int i = 0; i < n; ++i)
    if (!adm[i]) pruned[i] = 0;
  return KC_OK;
}

int32_t kc_sampler_generate_scan(kc_planner *p, const double vel[3], const double pose[3],
                                 const double *ranges, const double *angles, int32_t n,
                                 kc_samples *out) {
  KC_REQUIRE(p, KC_ERR_INVALID_ARG, "null handle");
  KC_REQUIRE(n == 0 || (ranges && angles), KC_ERR_INVALID_ARG, "null scan arrays");
  KC_TRY(kc::ensure_device());
  SensorDesc sd;
  sd.is_cloud = 0;
  sd.n = n;
  sd.host = ranges;
  sd.host2 = angles;
  return run_sampler(p, vel, pose, sd, out);
}

int32_t kc_sampler_generate_cloud(kc_planner *p, const double vel[3], const double pose[3],
                                  const float *xyz, int32_t n, kc_samples *out) {
  KC_REQUIRE(p, KC_ERR_INVALID_ARG, "null handle");
  KC_REQUIRE(n == 0 || xyz, KC_ERR_INVALID_ARG, "null cloud");
  KC_TRY(kc::ensure_device());
  SensorDesc sd;
  sd.is_cloud = 1;
  sd.n = n;
  sd.host = xyz;
  return run_sampler(p, vel, pose, sd, out);
}

// ---- CostEvaluator API ----------------------------------------------------------------------
int32_t kc_cost_set_points_scan(kc_planner *p, const double *ranges, const double *angles,
                                int32_t n, const double pose[3], float max_sensor_range,
                                float multiple) {
  KC_REQUIRE(p && pose, KC_ERR_INVALID_ARG, "null argument");
  KC_REQUIRE(n >= 0 && (n == 0 || (ranges && angles)), KC_ERR_INVALID_ARG, "bad scan arrays");
  KC_TRY(kc::ensure_device());
  p->cost_sensor.resize((size_t)n * 16);
  if (n) {
    memcpy(p->cost_sensor.data(), ranges, (size_t)n * 8);
    memcpy(p->cost_sensor.data() + (size_t)n * 8, angles, (size_t)n * 8);
  }
  p->cost_sensor_is_cloud = 0;
  p->cost_sensor_n = n;
  memcpy(p->cost_pose, pose, sizeof(p->cost_pose));
  p->cost_D = max_sensor_range / multiple;
  return KC_OK;
}

int32_t kc_cost_set_points_cloud(kc_planner *p, const float *xyz, int32_t n, const double pose[3],
                                 float max_sensor_range, float multiple) {
  KC_REQUIRE(p && pose, KC_ERR_INVALID_ARG, "null argument");
  KC_REQUIRE(n >= 0 && (n == 0 || xyz), KC_ERR_INVALID_ARG, "bad cloud");
  KC_TRY(kc::ensure_device());
  p->cost_sensor.resize((size_t)n * 12);
  if (n) memcpy(p->cost_sensor.data(), xyz, (size_t)n * 12);
  p->cost_sensor_is_cloud = 1;
  p->cost_sensor_n = n;
  memcpy(p->cost_pose, pose, sizeof(p->cost_pose));
  p->cost_D = max_sensor_range / multiple;
  return KC_OK;
}

int32_t kc_cost_evaluate(kc_planner *p, int32_t n_traj, int32_t P, const float *vx, const float *vy,
                         const float *omega, const float *x, const float *y, int32_t seg_start,
                         int32_t seg_count, const double *custom, int32_t n_custom,
                         float *costs_out, kc_cycle_result *out) {
  KC_REQUIRE(p && out, KC_ERR_INVALID_ARG, "null argument");
  KC_REQUIRE(n_traj >= 0 && P >= 2, KC_ERR_INVALID_ARG, "bad sample batch shape");
  KC_REQUIRE(n_traj == 0 || (vx && vy && omega && x && y), KC_ERR_INVALID_ARG, "null sample arrays");
  KC_REQUIRE(p->path_n >= 2, KC_ERR_INVALID_ARG, "reference path not set");
  KC_REQUIRE(n_custom >= 0 && (n_custom == 0 || custom), KC_ERR_INVALID_ARG, "bad custom cost terms");
  KC_TRY(kc::ensure_device());
  if (n_custom == 0) custom = nullptr;
  memset(out, 0, sizeof(*out));
  out->n_points = P;
  if (n_traj == 0) return KC_OK;
  const int savedP = p->P;
  p->P = P;
  struct Restore {
    kc_planner *p;
    int P;
    ~Restore() { p->P = P; }
  } restore{p, savedP};

  const size_t nv = (size_t)n_traj * (P - 1), np = (size_t)n_traj * P;
  const size_t cu_off = (3 * nv + 2 * np + 3) & ~(size_t)3;  // doubles start 16-byte aligned
  const size_t ncu = (size_t)n_traj * (size_t)n_custom;
  KC_TRY(p->d_in.reserve(cu_off + 2 * ncu + 16));
  float *dvx = p->d_in.ptr, *dvy = dvx + nv, *dom = dvy + nv, *dx = dom + nv, *dy = dx + np;
  double *dcu = reinterpret_cast<double *>(p->d_in.ptr + cu_off);
  cudaStream_t st = p->stream;
  KC_TRY(upload_pageable(p, {{dx, x, np * 4}, {dy, y, np * 4}, {dvx, vx, nv * 4}, {dvy, vy, nv * 4},
                             {dom, omega, nv * 4}, {dcu, custom, custom ? ncu * 8 : 0}}, st));

  SensorDesc sd;
  sd.is_cloud = p->cost_sensor_is_cloud;
  sd.n = p->cost_sensor_n;
  sd.host = p->cost_sensor.data();
  sd.host2 = p->cost_sensor.data() + (size_t)p->cost_sensor_n * 8;
  Axes ax;  // no velocity slots in this mode
  ax.row_off.push_back(0);
  RobotCtx cx;
  Sizes sz;
  const double zero3[3] = {0, 0, 0};
  KC_TRY(fill_ctx_scalars(p, p->P, own_path(p), zero3, zero3, sd, seg_start, seg_count, false, true, p->cost_D,
                          p->cost_pose, ax, cx, sz));
  cx.n_traj = n_traj;
  cx.in_vx = dvx;
  cx.in_vy = dvy;
  cx.in_om = dom;
  cx.in_x = dx;
  cx.in_y = dy;
  cx.custom = custom ? dcu : nullptr;
  cx.n_custom = n_custom;

  if (cx.obs_enabled) {  // grid window = bounding box of the samples grown by the cost cut-off
    KC_TRY(p->d_bbox.reserve(4));
    const int init[4] = {host_float_to_ordered(FLT_MAX), host_float_to_ordered(-FLT_MAX),
                         host_float_to_ordered(FLT_MAX), host_float_to_ordered(-FLT_MAX)};
    KC_CUDA(cudaMemcpyAsync(p->d_bbox.ptr, init, sizeof(init), cudaMemcpyHostToDevice, st));
    const int gb = std::max(1, std::min((int)((np + 255) / 256), 4 * sm_count()));
    k_bbox<<<gb, 256, 0, st>>>(dx, dy, np, p->d_bbox.ptr);
    p->launches += 1;
    int bb[4];
    KC_CUDA(cudaMemcpyAsync(bb, p->d_bbox.ptr, sizeof(bb), cudaMemcpyDeviceToHost, st));
    KC_CUDA(cudaStreamSynchronize(st));
    const float mnx = ordered_to_float(bb[0]), mxx = ordered_to_float(bb[1]);
    const float mny = ordered_to_float(bb[2]), mxy = ordered_to_float(bb[3]);
    if (!(mnx <= mxx && mny <= mxy)) {
      cx.obs_enabled = 0;  // no finite trajectory point: the term can never win a '<'
    } else {
      const double qhalf = 0.5 * std::max((double)mxx - mnx, (double)mxy - mny) * 1.001 + 1e-3;
      const double half = qhalf + (double)p->cost_D * 1.001 + 1e-3;
      set_grid_window(cx, 0.5f * (mnx + mxx), 0.5f * (mny + mxy), half, qhalf);
    }
  }
  const size_t zw = zero_words_per_robot(0);
  KC_TRY(reserve_workspace(p, 1, zw, 0, sd.n, n_traj, P));
  bind_workspace(p, cx, own_path(p), 0, zw, 0, 0, sd.n, n_traj, P);
  SensorDesc sdl = sd;
  const StageLayout L = plan_stage(ax, sdl);
  KC_TRY(p->h_stage.reserve(L.total));
  KC_TRY(p->d_stage.reserve(L.total));
  uint8_t *hs = p->h_stage.ptr, *ds = p->d_stage.ptr;
  cx.sensor = ds + L.sensor_off;
  memcpy(hs + L.ctx_off, &cx, sizeof(cx));
  if (sd.n > 0)
    memcpy(hs + L.sensor_off, p->cost_sensor.data(), sd.is_cloud ? (size_t)sd.n * 12 : (size_t)sd.n * 16);
  KC_CUDA(cudaMemcpyAsync(ds, hs, L.total, cudaMemcpyHostToDevice, st));
  const RobotCtx *d_ctx = reinterpret_cast<const RobotCtx *>(ds);
  if (cx.obs_enabled) {
    KC_CUDA(cudaMemsetAsync(p->d_zero.ptr, 0, zw * 4, st));
    const int gx = std::max(1, std::min((sd.n + 255) / 256, 8 * sm_count()));
    k_prep_points<<<dim3(gx, 1), 256, 0, st>>>(d_ctx);
    k_scan_dist<<<dim3(kScanBlocks, 1), 1024, 0, st>>>(d_ctx);
    const int n_class = class_ctas_for(qcells(cx));
    k_scatter<<<dim3(gx + n_class, 1), 256, 0, st>>>(d_ctx, n_class);
    k_cell_cand<<<dim3((qcells(cx) + kCandWarps - 1) / kCandWarps, 1), kCandWarps * 32, 0, st>>>(d_ctx);
    p->launches += 4;
  }
  size_t smem;
  const int warps = pick_eval_warps(P, cx.seg_count, 0, smem);
  KC_TRY(allow_smem(k_eval_rows, smem));
  k_eval_rows<<<dim3((n_traj + warps - 1) / warps, 1), warps * 32, smem, st>>>(d_ctx);
  k_select<<<dim3(1, 1), 1024, 0, st>>>(d_ctx);
  p->launches += 2;
  KC_CUDA(cudaGetLastError());
  KC_TRY(p->h_costs.reserve(n_traj));
  KC_CUDA(cudaMemcpyAsync(p->h_result.ptr, p->d_result.ptr, sizeof(ResultHeader),
                          cudaMemcpyDeviceToHost, st));
  if (costs_out)
    KC_CUDA(cudaMemcpyAsync(p->h_costs.ptr, p->d_costs.ptr, (size_t)n_traj * 4, cudaMemcpyDeviceToHost, st));
  KC_CUDA(cudaStreamSynchronize(st));
  if (costs_out) memcpy(costs_out, p->h_costs.ptr, (size_t)n_traj * 4);
  const ResultHeader *h = reinterpret_cast<const ResultHeader *>(p->h_result.ptr);
  out->found = h->found;
  out->cost = h->cost;
  out->slot = h->slot;
  out->n_slots = n_traj;
  out->n_admissible = n_traj;
  if (h->found) {  // winner row = the caller's own row (TrajSearchResult holds a copy of it)
    float *rows = reinterpret_cast<float *>(p->h_result.ptr + sizeof(ResultHeader));
    const size_t w = (size_t)h->slot;
    memcpy(rows, vx + w * (P - 1), (size_t)(P - 1) * 4);
    memcpy(rows + (P - 1), vy + w * (P - 1), (size_t)(P - 1) * 4);
    memcpy(rows + 2 * (P - 1), omega + w * (P - 1), (size_t)(P - 1) * 4);
    memcpy(rows + 3 * (P - 1), x + w * P, (size_t)P * 4);
    memcpy(rows + 3 * (P - 1) + P, y + w * P, (size_t)P * 4);
    out->vx = rows;
    out->vy = rows + (P - 1);
    out->omega = rows + 2 * (P - 1);
    out->x = rows + 3 * (P - 1);
    out->y = rows + 3 * (P - 1) + P;
  }
  p->last_slots = n_traj;
  p->last_was_cycle = false;
  return KC_OK;
}

// ---- device-resident replay ------------------------------------------------------------------
int32_t kc_planner_bank_alloc(kc_planner *p, int32_t n_slots, int32_t max_points) {
  KC_REQUIRE(p && n_slots > 0 && max_points > 0, KC_ERR_INVALID_ARG, "bad bank shape");
  KC_TRY(kc::ensure_device());
  KC_TRY(p->d_bank.reserve((size_t)n_slots * max_points * 3));
  p->bank_slots = n_slots;
  p->bank_max = max_points;
  p->bank_counts.assign(n_slots, 0);
  return KC_OK;
}

int32_t kc_planner_bank_upload(kc_planner *p, int32_t slot, const float *xyz, int32_t n) {
  KC_REQUIRE(p && xyz, KC_ERR_INVALID_ARG, "null argument");
  KC_REQUIRE(slot >= 0 && slot < p->bank_slots && n >= 0 && n <= p->bank_max, KC_ERR_OUT_OF_RANGE,
             "bank slot/size out of range");
  KC_TRY(kc::ensure_device());
  KC_CUDA(cudaMemcpy(p->d_bank.ptr + (size_t)slot * p->bank_max * 3, xyz, (size_t)n * 12,
                     cudaMemcpyHostToDevice));
  p->bank_counts[slot] = n;
  return KC_OK;
}

int32_t kc_planner_replay(kc_planner *p, int32_t first_slot, int32_t n_cycles, const double vel[3],
                          const double pose[3], int32_t seg_start, int32_t seg_count,
                          float *total_ms, float *eval_ms, kc_cycle_result *last) {
  KC_REQUIRE(p && vel && pose && n_cycles > 0, KC_ERR_INVALID_ARG, "bad replay arguments");
  KC_REQUIRE(p->bank_slots > 0, KC_ERR_INVALID_ARG, "no cloud bank allocated");
  KC_REQUIRE(p->path_n >= 2, KC_ERR_INVALID_ARG, "reference path not set");
  KC_TRY(kc::ensure_device());
  p->heavy_bound = p->heavy_kernel_on();
  p->general_bound = false;  // clouds are world-frame data: identity octree frame
  Axes ax;
  enumerate_axes(p->cfg, vel, ax);
  const float D = p->cfg.max_local_range / 3.0f;
  // one ctx per distinct bank slot, uploaded once before the timed region
  const int ns = p->bank_slots;
  std::vector<RobotCtx> ctxs(ns);
  Sizes szmax;
  int32_t max_sensor = 0;
  for (int s = 0; s < ns; ++s) {
    SensorDesc sd;
    sd.is_cloud = 1;
    sd.n = p->bank_counts[s];
    Sizes sz;
    KC_TRY(fill_ctx_scalars(p, p->P, own_path(p), vel, pose, sd, seg_start, seg_count, true, true, D, pose, ax,
                            ctxs[s], sz));
    const double reach = ax.max_speed * (double)(p->P - 1) * ctxs[s].dt * 1.001 + 1e-3;
    set_grid_window(ctxs[s], (float)pose[0], (float)pose[1], reach + (double)D * 1.001 + 1e-3, reach + 1e-3);
    szmax.bitmap_words = std::max(szmax.bitmap_words, sz.bitmap_words);
    szmax.sph_words = std::max(szmax.sph_words, sz.sph_words);
    max_sensor = std::max(max_sensor, sd.n);
  }
  const size_t zw = zero_words_per_robot(szmax.bitmap_words);
  KC_TRY(reserve_workspace(p, 1, zw, szmax.sph_words, max_sensor, ax.n_slots, p->P));
  SensorDesc none;
  none.dev = p->d_bank.ptr;
  none.n = 0;
  StageLayout L = plan_stage(ax, none);
  const size_t ctx_bytes = align_up(sizeof(RobotCtx) * (size_t)ns);
  const size_t total = ctx_bytes + L.total;
  KC_TRY(p->h_stage.reserve(total));
  KC_TRY(p->d_stage.reserve(total));
  uint8_t *hs = p->h_stage.ptr, *ds = p->d_stage.ptr;
  const size_t shift = ctx_bytes - L.vx_off;  // axes follow the ctx array
  int32_t dil_words = 0;
  for (int s = 0; s < ns; ++s) {
    RobotCtx &cx = ctxs[s];
    bind_workspace(p, cx, own_path(p), 0, zw, szmax.bitmap_words, szmax.sph_words, max_sensor, ax.n_slots, p->P);
    dil_words = std::max(dil_words, plan_dilation(cx, (size_t)cx.bm_rows * cx.bm_wpr));
    cx.ax_vx = reinterpret_cast<const double *>(ds + L.vx_off + shift);
    cx.ax_vy = reinterpret_cast<const double *>(ds + L.vy_off + shift);
    cx.ax_om = reinterpret_cast<const double *>(ds + L.om_off + shift);
    cx.row_off = reinterpret_cast<const int32_t *>(ds + L.row_off + shift);
    cx.sensor = p->d_bank.ptr + (size_t)s * p->bank_max * 3;
    memcpy(hs + sizeof(RobotCtx) * (size_t)s, &cx, sizeof(cx));
  }
  if (!ax.vx.empty()) memcpy(hs + L.vx_off + shift, ax.vx.data(), ax.vx.size() * 8);
  if (!ax.vy.empty()) memcpy(hs + L.vy_off + shift, ax.vy.data(), ax.vy.size() * 8);
  if (!ax.om.empty()) memcpy(hs + L.om_off + shift, ax.om.data(), ax.om.size() * 8);
  memcpy(hs + L.row_off + shift, ax.row_off.data(), ax.row_off.size() * 4);
  KC_CUDA(cudaMemcpyAsync(ds, hs, total, cudaMemcpyHostToDevice, p->stream));
  KC_CUDA(cudaStreamSynchronize(p->stream));
  const RobotCtx *d_ctx = reinterpret_cast<const RobotCtx *>(ds);

  const bool time_eval = eval_ms != nullptr;
  if (time_eval) {
    while ((int)p->evk.size() < 2 * n_cycles) {
      cudaEvent_t e;
      KC_CUDA(cudaEventCreate(&e));
      p->evk.push_back(e);
    }
  }
  // one graph per distinct resident cloud; a larger bank would thrash the cache: plain launches
  const bool saved_graphs = p->use_graphs;
  if (ns > kc_planner::kGraphSlots) p->use_graphs = false;
  struct RestoreGraphs {
    kc_planner *p;
    bool v;
    ~RestoreGraphs() { p->use_graphs = v; }
  } restore_graphs{p, saved_graphs};
  KC_CUDA(cudaEventRecord(p->ev0, p->stream));
  for (int i = 0; i < n_cycles; ++i) {
    const int s = ((first_slot + i) % ns + ns) % ns;
    KC_TRY(launch_cycle(p, d_ctx + s, 1, zw, szmax.sph_words, p->bank_counts[s], ax.n_slots, p->P,
                        ctxs[s].seg_count, p->bank_counts[s] > 0, 0,
                        time_eval ? p->evk[2 * i] : nullptr, time_eval ? p->evk[2 * i + 1] : nullptr,
                        qcells(ctxs[s]), dil_words));
  }
  KC_CUDA(cudaEventRecord(p->ev1, p->stream));
  KC_CUDA(cudaStreamSynchronize(p->stream));
  float ms = 0.0f;
  KC_CUDA(cudaEventElapsedTime(&ms, p->ev0, p->ev1));
  if (total_ms) *total_ms = ms;
  if (time_eval) {
    double acc = 0.0;
    for (int i = 0; i < n_cycles; ++i) {
      float m = 0.0f;
      KC_CUDA(cudaEventElapsedTime(&m, p->evk[2 * i], p->evk[2 * i + 1]));
      acc += m;
    }
    *eval_ms = (float)acc;
  }
  p->last_slots = ax.n_slots;
  p->last_was_cycle = true;
  p->last_replay = true;
  if (last) {
    const size_t res_bytes = sizeof(ResultHeader) + sizeof(float) * 5 * (size_t)p->P;
    KC_CUDA(cudaMemcpy(p->h_result.ptr, p->d_result.ptr, res_bytes, cudaMemcpyDeviceToHost));
    fill_result(p, p->h_result.ptr, p->P, ax.n_slots, last);
  }
  return KC_OK;
}

int64_t kc_planner_launch_count(const kc_planner *p) { return p ? p->launches : 0; }

// page-locked host memory for callers that want their sensor buffers DMA-ed without a staging copy
void *kc_pinned_alloc(size_t bytes) {
  if (ensure_device() != KC_OK) return nullptr;
  void *q = nullptr;
  if (cudaHostAlloc(&q, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
    cudaGetLastError();
    set_error("cudaHostAlloc of %zu bytes failed", bytes);
    return nullptr;
  }
  return q;
}
void kc_pinned_free(void *q) {
  if (q) cudaFreeHost(q);
}

int32_t kc_planner_set_tuning(kc_planner *p, int32_t key, int64_t value) {
  KC_REQUIRE(p, KC_ERR_INVALID_ARG, "null handle");
  KC_REQUIRE(key >= 0 && key <= 13, KC_ERR_INVALID_ARG, "unknown tuning key %d", key);
  KC_TRY(kc::ensure_device());
  if (key == 8) {
    p->poll_result = value != 0;
    return KC_OK;
  }
  // a switch can change the kernel set of a cycle: captured launch graphs are rebuilt on next use
  KC_CUDA(cudaStreamSynchronize(p->stream));
  for (kc_planner::GraphSlot &g : p->graphs) {
    if (g.exec) cudaGraphExecDestroy(g.exec);
    g.exec = nullptr;
  }
  if (key == 9) {
    p->use_pdl = value != 0;
    return KC_OK;
  }
  if (key == 13) {  // survivors up to which the exact stage works by (slot, point) pair
    KC_REQUIRE(value >= 0 && value <= (1 << 30), KC_ERR_OUT_OF_RANGE, "by-point limit out of range");
    p->by_point_max = (int32_t)value;
    return KC_OK;
  }
  if (key == 12) {  // robots per launch set of a batched sweep
    KC_REQUIRE(value >= 1 && value <= kBatchChunk, KC_ERR_OUT_OF_RANGE, "sweep chunk out of range [1, %d]", kBatchChunk);
    p->batch_chunk_max = (int32_t)value;
    return KC_OK;
  }
  if (key == 11) {  // per-cell candidate lists: 1 always (default), -1 only without branch and bound, 0 never
    KC_REQUIRE(value >= -1 && value <= 1, KC_ERR_OUT_OF_RANGE, "candidate-list mode out of range [-1, 1]");
    p->cand_lists = (int32_t)value;
    return KC_OK;
  }
  if (key == 10) {  // heavy-cell policy: -1 adaptive (default), 0 never, > 0 fixed threshold, kernel always on
    KC_REQUIRE(value >= -1 && value <= (1 << 30), KC_ERR_OUT_OF_RANGE, "heavy-cell threshold out of range");
    p->heavy_points = (int32_t)value;
    return KC_OK;
  }
  if (key == 7) {
    KC_REQUIRE(value >= 0 && value <= 2, KC_ERR_OUT_OF_RANGE, "branch-and-bound mode out of range [0, 2]");
    p->use_prune = (int32_t)value;
    return KC_OK;
  }
  if (key == 6) return KC_OK;  // retired (rows per warp of an earlier rollout kernel)
  if (key == 5) {
    p->use_reach_mask = value != 0;
    return KC_OK;
  }
  if (key == 4) {
    p->timeline = value != 0;
    return KC_OK;
  }
  if (key == 2) {
    p->zero_copy_cloud = value != 0;
    return KC_OK;
  }
  if (key == 3) {
    p->mapped_result = value != 0;
    return KC_OK;
  }
  if (key == 1) {  // 1 = replay the cycle's launch set as a CUDA graph (default), 0 = plain launches
    p->use_graphs = value != 0;
    return KC_OK;
  }
  KC_REQUIRE(value >= -1 && value <= (int64_t)kCandCap, KC_ERR_OUT_OF_RANGE,
             "candidate pool capacity out of range [-1, %d]", kCandCap);
  p->cand_cap = (int32_t)value;
  return KC_OK;
}

// developer timeline of the last plain-launch cycle (tuning key 4): for kernel i, names[i] and
// (start, end) in microseconds after the first recorded event; returns the kernel count
int32_t kc_planner_debug_timeline(kc_planner *p, const char **names, float *start_us, float *end_us,
                                  int32_t cap) {
  KC_REQUIRE(p && names && start_us && end_us, KC_ERR_INVALID_ARG, "null argument");
  KC_TRY(kc::ensure_device());
  KC_CUDA(cudaDeviceSynchronize());
  int n = 0;
  for (int i = 0; i < p->tl_n && i < cap; ++i) {
    float a = 0.0f, b = 0.0f;
    if (cudaEventElapsedTime(&a, p->tl_ev[0], p->tl_ev[2 * i]) != cudaSuccess ||
        cudaEventElapsedTime(&b, p->tl_ev[0], p->tl_ev[2 * i + 1]) != cudaSuccess) {
      cudaGetLastError();
      continue;
    }
    names[n] = p->tl_name[i];
    start_us[n] = a * 1e3f;
    end_us[n] = b * 1e3f;
    ++n;
  }
  return n;
}

// developer time stamps of k_cost_eval (library built with -DKC_DBG_STAMPS): reset before a cycle,
// read after it; out[i] in nanoseconds relative to out[0]
int32_t kc_planner_debug_stamps(kc_planner *p, int32_t reset, int64_t out[8]) {
  KC_REQUIRE(p, KC_ERR_INVALID_ARG, "null handle");
  KC_TRY(kc::ensure_device());
  KC_TRY(p->d_dbg.reserve(96));
  KC_CUDA(cudaDeviceSynchronize());
  if (reset > 0) {
    unsigned long long init[96];
    for (int i = 0; i < 96; ++i) init[i] = (i == 0 || i == 14 || (i >= 32 && i < 64 && !(i & 1))) ? ~0ull : 0ull;
    KC_CUDA(cudaMemcpy(p->d_dbg.ptr, init, sizeof(init), cudaMemcpyHostToDevice));
    return KC_OK;
  }
  unsigned long long v[96];
  KC_CUDA(cudaMemcpy(v, p->d_dbg.ptr, sizeof(v), cudaMemcpyDeviceToHost));
  if (reset < 0) {  // raw group -reset of eight (rollout phase sums / maxima; groups 4-7: the cycle timeline)
    for (int i = 0; i < 8 && out; ++i) out[i] = (int64_t)v[((-reset) % 12) * 8 + i];  // (-12: group 0)
    return KC_OK;
  }
  for (int i = 0; i < 8 && out; ++i) out[i] = (i >= 6) ? (int64_t)v[i] : (int64_t)(v[i] - v[0]);  // 6, 7: plain counters
  return KC_OK;
}

int32_t kc_planner_debug_stats(kc_planner *p, int64_t out[8]) {
  KC_REQUIRE(p && out, KC_ERR_INVALID_ARG, "null argument");
  KC_REQUIRE(p->last_was_cycle && p->last_ctx.cell_info, KC_ERR_INVALID_ARG, "no cycle has run");
  KC_TRY(kc::ensure_device());
  const RobotCtx &cx = p->last_ctx;
  for (int i = 0; i < 8; ++i) out[i] = 0;
  KC_CUDA(cudaStreamSynchronize(p->stream));
  if (!cx.obs_enabled) return KC_OK;
  std::vector<int4> info((size_t)kGridN * kGridN);
  int32_t used = 0, kept = 0;
  KC_CUDA(cudaMemcpy(info.data(), cx.cell_info, info.size() * sizeof(int4), cudaMemcpyDeviceToHost));
  KC_CUDA(cudaMemcpy(&used, cx.cand_ctr, 4, cudaMemcpyDeviceToHost));
  KC_CUDA(cudaMemcpy(&kept, cx.cell_start + kGridN * kGridN, 4, cudaMemcpyDeviceToHost));
  out[0] = used;
  out[5] = kept;
  if (cx.pcand_enabled) {
    std::vector<int2> pinfo((size_t)kGridN * kGridN);
    int32_t pused = 0;
    KC_CUDA(cudaMemcpy(pinfo.data(), cx.pcell_info, pinfo.size() * sizeof(int2), cudaMemcpyDeviceToHost));
    KC_CUDA(cudaMemcpy(&pused, cx.pcand_ctr, 4, cudaMemcpyDeviceToHost));
    out[6] = pused;
    for (int y = cx.q_y0; y <= cx.q_y1; ++y)
      for (int x = cx.q_x0; x <= cx.q_x1; ++x) out[7] = std::max<int64_t>(out[7], pinfo[(size_t)y * kGridN + x].y);
  }
  for (int y = cx.q_y0; y <= cx.q_y1; ++y)
    for (int x = cx.q_x0; x <= cx.q_x1; ++x) {
      const int4 ci = info[(size_t)y * kGridN + x];
      out[1] += 1;
      if (ci.z > 0) out[2] += 1;
      if (ci.z < 0) out[3] += 1;
      out[4] = std::max<int64_t>(out[4], ci.z);
    }
  return KC_OK;
}

// Brute-force evaluation of the obstacle term of the LAST kc_planner_cycle_* call: verification of
// the pruned nearest-obstacle search at full problem size and the FP32 roofline measurement. Not on
// the control path.
int32_t kc_planner_bruteforce_obstacle_costs(kc_planner *p, float *costs, float *pass1_ms,
                                             float *total_ms, double *pair_evaluations) {
  KC_REQUIRE(p && costs, KC_ERR_INVALID_ARG, "null argument");
  KC_REQUIRE(p->last_was_cycle && p->last_ctx.rows_x && !p->last_replay, KC_ERR_INVALID_ARG,
             "no kc_planner_cycle_* call has run on this handle");
  KC_TRY(kc::ensure_device());
  const RobotCtx &cx = p->last_ctx;
  const int n_slots = cx.n_slots, M = cx.n_sensor, P = cx.P;
  if (pass1_ms) *pass1_ms = 0.0f;
  if (total_ms) *total_ms = 0.0f;
  if (pair_evaluations) *pair_evaluations = 0.0;
  if (n_slots == 0) return KC_OK;
  cudaStream_t st = p->stream;
  KC_CUDA(cudaStreamSynchronize(st));
  const RobotCtx *d_ctx = reinterpret_cast<const RobotCtx *>(p->d_stage.ptr);
  int32_t n_list = 0;
  KC_CUDA(cudaMemcpy(&n_list, cx.n_list, 4, cudaMemcpyDeviceToHost));
  KC_TRY(p->d_bf_xy.reserve((size_t)std::max(M, 2) + 2));
  KC_TRY(p->d_bf_min.reserve(2 * (size_t)n_slots));
  KC_TRY(p->d_bf_cost.reserve((size_t)n_slots));
  unsigned int *min32 = p->d_bf_min.ptr, *min_exact = min32 + n_slots;
  KC_CUDA(cudaMemsetAsync(min32, 0x7f, 2 * (size_t)n_slots * 4, st));  // 3.39e38: "no finite pair"
  if (M > 0 && n_list > 0) {
    // KC_BF_SCALAR=1 selects the scalar-instruction form of the same arithmetic (A/B of the packed FP32 path)
    const char *bf_scalar = getenv("KC_BF_SCALAR");
    const bool packed = !(bf_scalar && bf_scalar[0] == '1');
    k_transform_points<<<std::max(1, std::min((M + 255) / 256, 8 * sm_count())), 256, 0, st>>>(d_ctx, p->d_bf_xy.ptr, packed ? 1 : 0);
    const long long total = (long long)n_list * P;
    const int entry_blocks = (int)((total + 2047) / 2048);
    const int all_tiles = (M + kBfTile - 1) / kBfTile;
    // enough work units for ~16 per SM, at least 2 tiles each
    int chunks = std::max(1, std::min(all_tiles / 2, (16 * sm_count() + entry_blocks - 1) / entry_blocks));
    const int tiles_per_chunk = (all_tiles + chunks - 1) / chunks;
    chunks = (all_tiles + tiles_per_chunk - 1) / tiles_per_chunk;
    const dim3 grid(entry_blocks, chunks);
    KC_CUDA(cudaEventRecord(p->ev0, st));
    if (packed)
      k_obstacle_bruteforce<false, true><<<grid, 256, 0, st>>>(d_ctx, p->d_bf_xy.ptr, M, tiles_per_chunk, min32, min_exact);
    else
      k_obstacle_bruteforce<false, false><<<grid, 256, 0, st>>>(d_ctx, p->d_bf_xy.ptr, M, tiles_per_chunk, min32, min_exact);
    KC_CUDA(cudaEventRecord(p->ev1, st));
    if (packed)
      k_obstacle_bruteforce<true, true><<<grid, 256, 0, st>>>(d_ctx, p->d_bf_xy.ptr, M, tiles_per_chunk, min32, min_exact);
    else
      k_obstacle_bruteforce<true, false><<<grid, 256, 0, st>>>(d_ctx, p->d_bf_xy.ptr, M, tiles_per_chunk, min32, min_exact);
    p->launches += 3;
    if (pair_evaluations) *pair_evaluations = (double)total * (double)M;
  }
  k_bruteforce_cost<<<(n_slots + 255) / 256, 256, 0, st>>>(d_ctx, min_exact, p->d_bf_cost.ptr);
  p->launches += 1;
  KC_CUDA(cudaGetLastError());
  KC_TRY(p->h_costs.reserve(n_slots));
  KC_CUDA(cudaMemcpyAsync(p->h_costs.ptr, p->d_bf_cost.ptr, (size_t)n_slots * 4, cudaMemcpyDeviceToHost, st));
  KC_CUDA(cudaStreamSynchronize(st));
  memcpy(costs, p->h_costs.ptr, (size_t)n_slots * 4);
  if (M > 0 && n_list > 0) {
    float ms = 0.0f;
    KC_CUDA(cudaEventElapsedTime(&ms, p->ev0, p->ev1));
    if (pass1_ms) *pass1_ms = ms;
  }
  (void)total_ms;
  return KC_OK;
}

}  // extern "C"

// ---- batched multi-robot sweep ---------------------------------------------------------------
// The sweep runs chunk after chunk of kBatchChunk robots: one launch set per chunk (blockIdx.y =
// robot within the chunk) on a workspace sized for one chunk, so device memory stays bounded
// (~18 MB per robot of the chunk instead of per robot of the sweep) and the sensor data of chunk k+1
// is uploaded while chunk k computes.
//
// Robots of one launch set may differ in points per trajectory (P: a horizon shortened on path
// curvature), tracked segment length (S: near the path end), velocity slots and sensor count. Every
// kernel takes these bounds from its robot's ctx; the launch geometry takes the chunk's largest P and
// S only to size the per-warp shared-memory carve-outs and the warp count, which a smaller robot
// then fills in part. The per-robot strides of the workspace (heading table, trajectory rows,
// result record) are set by the largest P of the whole batch.

namespace {

int32_t batch_launch_chunk(kc_planner *p, int ci) {
  const int c0 = p->batch_starts[ci], Rc = p->batch_starts[ci + 1] - c0;
  const RobotCtx *d_ctx = reinterpret_cast<const RobotCtx *>(p->d_batch_stage.ptr) + c0;
  return launch_cycle(p, d_ctx, Rc, p->batch_zero_words * (size_t)Rc, p->batch_sph_words * (size_t)Rc,
                      p->batch_max_sensor, p->batch_max_slots, p->batch_chunk_P[ci], p->batch_chunk_S[ci],
                      p->batch_max_sensor > 0, 0, nullptr, nullptr, p->batch_max_qcells,
                      p->batch_dil_words);
}

int32_t batch_launch(kc_planner *p) {
  for (size_t ci = 0; ci + 1 < p->batch_starts.size(); ++ci) KC_TRY(batch_launch_chunk(p, (int)ci));
  return KC_OK;
}

// results [R]; cycles [R] or NULL: with cycles the whole records (header | rows) come back in one
// copy, without them only the R headers (strided gather)
int32_t batch_fetch(kc_planner *p, kc_batch_result *results, kc_cycle_result *cycles) {
  const int R = p->batch_R;
  const size_t res_bytes = align_up(sizeof(ResultHeader) + sizeof(float) * (5 * (size_t)p->batch_P));
  const size_t hstride = cycles ? res_bytes : sizeof(ResultHeader);
  if (cycles)
    KC_CUDA(cudaMemcpyAsync(p->h_result.ptr, p->d_result.ptr, (size_t)R * res_bytes, cudaMemcpyDeviceToHost,
                            p->stream));
  else  // strided gather of the R result headers: the only data that leaves the device
    KC_CUDA(cudaMemcpy2DAsync(p->h_result.ptr, sizeof(ResultHeader), p->d_result.ptr, res_bytes,
                              sizeof(ResultHeader), R, cudaMemcpyDeviceToHost, p->stream));
  KC_CUDA(cudaStreamSynchronize(p->stream));
  p->heavy_seen = false;
  for (int r = 0; r < R; ++r) {
    uint8_t *rec = p->h_result.ptr + (size_t)r * hstride;
    const RobotCtx &cx = p->batch_ctx[r];
    // a robot without velocity slots has no launch work: its record is what a single cycle reports
    if (cycles && cx.n_slots == 0) memset(rec, 0, sizeof(ResultHeader) + sizeof(float) * 5 * (size_t)cx.P);
    const ResultHeader &h = *reinterpret_cast<const ResultHeader *>(rec);
    if (h.heavy_cells) p->heavy_seen = true;  // feedback for the next sweep's launch set
    results[r].found = h.n_admissible ? h.found : 0;
    results[r].cost = h.n_admissible ? h.cost : 0.0f;
    results[r].slot = h.slot;
    results[r].n_admissible = h.n_admissible;
    results[r].n_slots = cx.n_slots;
    if (cycles) {
      const bool heavy = p->heavy_seen;
      fill_result(p, rec, cx.P, cx.n_slots, &cycles[r]);
      p->heavy_seen = heavy;
    }
  }
  return KC_OK;
}

}  // namespace

namespace kc {

int32_t horizon_points(double time_step, double base_horizon, double &horizon) {
  const double min_h = 2.0 * time_step;  // trajectory_sampler.cpp:316-326
  if (horizon < min_h) horizon = min_h;
  if (horizon > base_horizon) horizon = base_horizon;
  return (int32_t)(size_t)(horizon / time_step);
}

int32_t planner_batch(kc_planner *p, int32_t R, const BatchRobot *rb, const BatchSensor &sen,
                      kc_batch_result *results, kc_cycle_result *cycles) {
  KC_REQUIRE(p && rb && results, KC_ERR_INVALID_ARG, "null argument");
  KC_REQUIRE(R > 0, KC_ERR_INVALID_ARG, "n_robots must be positive");
  KC_TRY(kc::ensure_device());
  const bool timing = getenv("KC_BATCH_TIMING") != nullptr;  // developer: host-side split on stderr
  const auto t_begin = std::chrono::steady_clock::now();
  auto since = [&] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(); };
  p->heavy_bound = p->batch_heavy = p->heavy_kernel_on();
  const float D = p->cfg.max_local_range / 3.0f;
  std::vector<Axes> axes(R);
  p->batch_ctx.assign(R, RobotCtx());
  Sizes szmax;
  int32_t max_sensor = 0, max_slots = 0, Pmax = 0;
  int64_t total_pts = 0, scan_total = 0;
  for (int r = 0; r < R; ++r) {
    KC_REQUIRE(rb[r].count >= 0 && rb[r].offset >= 0, KC_ERR_INVALID_ARG, "robot %d: bad sensor extents", r);
    KC_REQUIRE(rb[r].vel && rb[r].pose, KC_ERR_INVALID_ARG, "robot %d: null velocity or pose", r);
    KC_REQUIRE(rb[r].P >= 2, KC_ERR_INVALID_ARG, "robot %d: %d points per trajectory", r, rb[r].P);
    KC_REQUIRE(rb[r].path.n >= 2 && rb[r].path.hX && rb[r].path.hY && rb[r].path.dX, KC_ERR_INVALID_ARG,
               "robot %d: reference path not set", r);
    total_pts = std::max<int64_t>(total_pts, rb[r].offset + rb[r].count);
    scan_total += 2 * (int64_t)rb[r].count;
    Pmax = std::max(Pmax, rb[r].P);
  }
  if (sen.cloud)
    KC_REQUIRE(total_pts == 0 || sen.xyz, KC_ERR_INVALID_ARG, "null cloud");
  else
    KC_REQUIRE(total_pts == 0 || (sen.ranges && sen.angles), KC_ERR_INVALID_ARG, "null scan arrays");
  size_t axes_bytes = 0;
  bool general = false;
  for (int r = 0; r < R; ++r) {
    const BatchRobot &b = rb[r];
    enumerate_axes(p->cfg, b.vel, axes[r]);
    SensorDesc sd;
    sd.is_cloud = sen.cloud ? 1 : 0;
    sd.n = b.count;
    Sizes sz;
    RobotCtx &cx = p->batch_ctx[r];
    KC_TRY(fill_ctx_scalars(p, b.P, b.path, b.vel, b.pose, sd, b.seg_start, b.seg_count, true, true, D, b.pose,
                            axes[r], cx, sz));
    // clouds arrive in the world frame (identity octree frame); a scan's frame follows its robot's pose
    // through the shared mount, so whether it is tilted is the same for every robot
    if (r == 0) general = cx.coll_general != 0;
    KC_REQUIRE((cx.coll_general != 0) == general, KC_ERR_UNSUPPORTED, "mixed sensor frames in one batch");
    const double reach = axes[r].max_speed * (double)(b.P - 1) * cx.dt * 1.001 + 1e-3;
    set_grid_window(cx, (float)b.pose[0], (float)b.pose[1], reach + (double)D * 1.001 + 1e-3, reach + 1e-3);
    szmax.bitmap_words = std::max(szmax.bitmap_words, sz.bitmap_words);
    szmax.sph_words = std::max(szmax.sph_words, sz.sph_words);
    max_sensor = std::max(max_sensor, sd.n);
    max_slots = std::max(max_slots, axes[r].n_slots);
    axes_bytes += align_up((axes[r].vx.size() + axes[r].vy.size() + axes[r].om.size()) * 8 +
                           axes[r].row_off.size() * 4 + 64);
  }
  p->general_bound = p->batch_general = general;
  const size_t zw = zero_words_per_robot(szmax.bitmap_words);
  const int C = std::min(R, std::max(1, std::min(p->batch_chunk_max, kBatchChunk)));
  // chunk boundaries: the first chunk's clouds cannot be uploaded behind any computation, so the sweep
  // starts with small chunks (8, 16, 32 robots) and grows to kBatchChunk: the un-overlapped prologue
  // shrinks from 77 MB to 10 MB of host->device traffic
  p->batch_starts.clear();
  for (int c0 = 0, step = std::min(8, C); c0 < R; c0 += step, step = std::min(2 * step, C)) p->batch_starts.push_back(c0);
  p->batch_starts.push_back(R);
  const size_t n_chunks = p->batch_starts.size() - 1;
  p->batch_chunk_P.assign(n_chunks, 0);
  p->batch_chunk_S.assign(n_chunks, 0);
  std::vector<int> slot_of(R);
  for (size_t c = 0; c < n_chunks; ++c)
    for (int r = p->batch_starts[c]; r < p->batch_starts[c + 1]; ++r) {
      slot_of[r] = r - p->batch_starts[c];
      p->batch_chunk_P[c] = std::max(p->batch_chunk_P[c], rb[r].P);
      p->batch_chunk_S[c] = std::max(p->batch_chunk_S[c], p->batch_ctx[r].seg_count);
    }
  KC_TRY(reserve_workspace(p, C, zw, szmax.sph_words, max_sensor, max_slots, Pmax));
  {
    const size_t res_bytes = align_up(sizeof(ResultHeader) + sizeof(float) * (5 * (size_t)Pmax));
    KC_TRY(p->d_result.reserve((size_t)R * res_bytes));
    KC_TRY(p->h_result.reserve((size_t)R * res_bytes));
  }
  std::vector<int64_t> scan_off;
  if (sen.cloud) {
    KC_TRY(p->d_batch_xyz.reserve((size_t)std::max<int64_t>(total_pts, 1) * 3));
  } else {
    KC_TRY(p->d_batch_scan.reserve((size_t)std::max<int64_t>(scan_total, 1)));
    KC_TRY(p->h_batch_scan.reserve((size_t)std::max<int64_t>(scan_total, 1)));
    scan_off.assign(R + 1, 0);
    for (int r = 0; r < R; ++r) scan_off[r + 1] = scan_off[r] + 2 * (int64_t)rb[r].count;
  }
  if (!p->copy) {
    KC_CUDA(cudaStreamCreateWithFlags(&p->copy, cudaStreamNonBlocking));
    KC_CUDA(cudaEventCreateWithFlags(&p->ev_copy, cudaEventDisableTiming));
  }
  const size_t ctx_bytes = align_up(sizeof(RobotCtx) * (size_t)R);
  KC_TRY(p->h_stage.reserve(ctx_bytes + axes_bytes));
  KC_TRY(p->d_batch_stage.reserve(ctx_bytes + axes_bytes));
  uint8_t *hs = p->h_stage.ptr, *ds = p->d_batch_stage.ptr;
  size_t o = ctx_bytes;
  int32_t batch_dil = 0;
  for (int r = 0; r < R; ++r) {
    RobotCtx &cx = p->batch_ctx[r];
    const Axes &a = axes[r];
    bind_workspace(p, cx, rb[r].path, slot_of[r], zw, szmax.bitmap_words, szmax.sph_words, max_sensor, max_slots,
                   Pmax, r);
    if (szmax.bitmap_words <= kDilMaxWords)  // every robot's bitmap must fit the shared smem carve-out
      batch_dil = std::max(batch_dil, plan_dilation(cx, (size_t)cx.bm_rows * cx.bm_wpr));
    cx.ax_vx = reinterpret_cast<const double *>(ds + o);
    if (!a.vx.empty()) memcpy(hs + o, a.vx.data(), a.vx.size() * 8);
    o += a.vx.size() * 8;
    cx.ax_vy = reinterpret_cast<const double *>(ds + o);
    if (!a.vy.empty()) memcpy(hs + o, a.vy.data(), a.vy.size() * 8);
    o += a.vy.size() * 8;
    cx.ax_om = reinterpret_cast<const double *>(ds + o);
    if (!a.om.empty()) memcpy(hs + o, a.om.data(), a.om.size() * 8);
    o += a.om.size() * 8;
    cx.row_off = reinterpret_cast<const int32_t *>(ds + o);
    memcpy(hs + o, a.row_off.data(), a.row_off.size() * 4);
    o = align_up(o + a.row_off.size() * 4);
    if (sen.cloud)
      cx.sensor = p->d_batch_xyz.ptr + 3 * rb[r].offset;
    else  // k_prep_points reads a scan as ranges [n] then angles [n]
      cx.sensor = p->d_batch_scan.ptr + scan_off[r];
    memcpy(hs + sizeof(RobotCtx) * (size_t)r, &cx, sizeof(cx));
  }
  KC_CUDA(cudaMemcpyAsync(ds, hs, o, cudaMemcpyHostToDevice, p->stream));
  p->batch_R = R;
  p->batch_chunk = C;
  p->batch_P = Pmax;
  p->batch_zero_words = zw;
  p->batch_sph_words = szmax.sph_words;
  p->batch_max_sensor = max_sensor;
  p->batch_max_slots = max_slots;
  p->batch_dil_words = batch_dil;
  p->batch_max_qcells = 0;
  for (int r = 0; r < R; ++r) p->batch_max_qcells = std::max(p->batch_max_qcells, qcells(p->batch_ctx[r]));
  // chunk pipeline: the copy stream uploads the sensor data chunk k needs (a page-locked caller cloud
  // is DMA-ed directly; pageable memory is staged by the driver, scans through the handle's page-locked
  // buffer, while the GPU works on the previous chunk), the compute stream waits for it and runs chunk k
  const double t_prep = since();
  int64_t up_lo = 0, up_hi = 0;  // point range already uploaded
  for (size_t ci = 0; ci < n_chunks; ++ci) {
    const int c0 = p->batch_starts[ci], c1 = p->batch_starts[ci + 1];
    if (sen.cloud) {
      int64_t lo = INT64_MAX, hi = 0;
      for (int r = c0; r < c1; ++r) {
        if (rb[r].count == 0) continue;
        lo = std::min<int64_t>(lo, rb[r].offset);
        hi = std::max<int64_t>(hi, rb[r].offset + rb[r].count);
      }
      if (lo < hi && !(lo >= up_lo && hi <= up_hi)) {
        int64_t a = lo, b = hi;
        if (up_lo < up_hi && lo >= up_lo && lo <= up_hi) {  // extends the uploaded range upwards
          a = up_hi;
          up_hi = hi;
        } else {  // disjoint layout: restart the bookkeeping with this range
          up_lo = lo;
          up_hi = hi;
        }
        if (a < b)
          KC_CUDA(cudaMemcpyAsync(p->d_batch_xyz.ptr + 3 * a, sen.xyz + 3 * a, (size_t)(b - a) * 12,
                                  cudaMemcpyHostToDevice, p->copy));
      }
    } else if (scan_off[c1] > scan_off[c0]) {
      double *h = p->h_batch_scan.ptr;
      for (int r = c0; r < c1; ++r) {
        const size_t n = (size_t)rb[r].count;
        if (!n) continue;
        memcpy(h + scan_off[r], sen.ranges + rb[r].offset, n * 8);
        memcpy(h + scan_off[r] + n, sen.angles + rb[r].offset, n * 8);
      }
      KC_CUDA(cudaMemcpyAsync(p->d_batch_scan.ptr + scan_off[c0], h + scan_off[c0],
                              (size_t)(scan_off[c1] - scan_off[c0]) * 8, cudaMemcpyHostToDevice, p->copy));
    }
    KC_CUDA(cudaEventRecord(p->ev_copy, p->copy));
    KC_CUDA(cudaStreamWaitEvent(p->stream, p->ev_copy, 0));
    KC_TRY(batch_launch_chunk(p, (int)ci));
  }
  const double t_enq = since();
  const int32_t rc = batch_fetch(p, results, cycles);
  if (timing)
    fprintf(stderr, "[kc batch] R=%d chunks=%zu host prep %.3f ms, enqueue %.3f ms, wait+fetch %.3f ms\n", R,
            n_chunks, t_prep, t_enq - t_prep, since() - t_enq);
  return rc;
}

}  // namespace kc

extern "C" {

int32_t kc_planner_batch_cloud(kc_planner *p, int32_t R, const double *vel, const double *pose,
                               const float *xyz, const int64_t *offsets, const int32_t *counts,
                               int32_t seg_start, int32_t seg_count, kc_batch_result *results) {
  KC_REQUIRE(p && vel && pose && offsets && counts && results, KC_ERR_INVALID_ARG, "null argument");
  KC_REQUIRE(R > 0, KC_ERR_INVALID_ARG, "n_robots must be positive");
  KC_REQUIRE(p->path_n >= 2, KC_ERR_INVALID_ARG, "reference path not set");
  KC_TRY(kc::ensure_device());
  std::vector<BatchRobot> rb(R);
  const BatchPath path = own_path(p);
  for (int r = 0; r < R; ++r) {
    KC_REQUIRE(counts[r] >= 0 && offsets[r] >= 0, KC_ERR_INVALID_ARG, "bad cloud extents");
    rb[r].vel = vel + 3 * r;
    rb[r].pose = pose + 3 * r;
    rb[r].P = p->P;
    rb[r].path = path;
    rb[r].seg_start = seg_start;
    rb[r].seg_count = seg_count;
    rb[r].offset = offsets[r];
    rb[r].count = counts[r];
  }
  BatchSensor sen;
  sen.cloud = true;
  sen.xyz = xyz;
  return planner_batch(p, R, rb.data(), sen, results, nullptr);
}

int32_t kc_planner_batch_replay(kc_planner *p, int32_t n_iters, float *total_ms,
                                kc_batch_result *results) {
  KC_REQUIRE(p && p->batch_R > 0 && n_iters > 0, KC_ERR_INVALID_ARG,
             "no resident batch (call kc_planner_batch_cloud first)");
  KC_TRY(kc::ensure_device());
  p->heavy_bound = p->batch_heavy;  // the resident ctxs were bound with this decision
  p->general_bound = p->batch_general;
  KC_CUDA(cudaEventRecord(p->ev0, p->stream));
  for (int i = 0; i < n_iters; ++i) KC_TRY(batch_launch(p));
  KC_CUDA(cudaEventRecord(p->ev1, p->stream));
  KC_CUDA(cudaStreamSynchronize(p->stream));
  float ms = 0.0f;
  KC_CUDA(cudaEventElapsedTime(&ms, p->ev0, p->ev1));
  if (total_ms) *total_ms = ms;
  if (results) return batch_fetch(p, results, nullptr);
  return KC_OK;
}

}  // extern "C"

// =================================================================================================
// Stand-alone collision checker (SURVEY section 8 row f4): the reference's CollisionChecker as its other
// users see it (PurePursuit avoidance rollouts src/controllers/pure_pursuit.cpp:154-155, OMPL state
// validity src/planning/ompl.cpp:95-97, TrajectorySampler::checkStatesFeasibility
// src/utils/trajectory_sampler.cpp:378-408). Same voxel model and pose test as the DWA rollout kernel;
// the bitmap is built once per sensor update / window and reused by later checks it still covers.
// =================================================================================================
struct kc_collision {
  kc_planner_config cfg;  // only shape, dims, sensor pose and octree_resolution are read
  hm::Rigid sensor_tf_body, stw;  // stw = sensor_tf_world_ as of the last sensor update
  double state[3] = {0, 0, 0};
  cudaStream_t stream = nullptr;
  int32_t n_sensor = 0, is_cloud = 1;
  double res_data = 0.0;  // octree resolution the current sensor data was inserted with
  DevBuf<uint8_t> d_sensor;
  PinnedBuf<uint8_t> h_stage;
  DevBuf<uint32_t> d_bitmap, d_sph;
  DevBuf<double> d_states;
  DevBuf<uint8_t> d_out;
  DevBuf<RobotCtx> d_ctx;
  RobotCtx ctx;           // host copy of the ctx the cached bitmap was built with
  bool bitmap_valid = false;
};

namespace {
// (x, y)_lo..hi: bounding box of the query positions in the octree frame (planar frames);
// w*: the same box in the world frame (general frames: a cube window around its centre)
int32_t collision_prepare(kc_collision *h, double x_lo, double x_hi, double y_lo, double y_hi, double wx_lo,
                          double wx_hi, double wy_lo, double wy_hi) {
  RobotCtx &cx = h->ctx;
  const double wcx = 0.5 * (wx_lo + wx_hi), wcy = 0.5 * (wy_lo + wy_hi);
  const double wreach = 0.5 * std::hypot(wx_hi - wx_lo, wy_hi - wy_lo) + 1e-6;
  if (h->bitmap_valid) {  // does the cached window still cover every voxel these poses can touch?
    RobotCtx probe = cx;
    Sizes sz;
    kc_planner_config c = h->cfg;
    c.octree_resolution = h->res_data;
    if (cx.coll_general) {
      KC_TRY(fill_collision_window_general(c, wcx, wcy, wreach, probe, sz));
      if (probe.g_kx0 >= cx.g_kx0 && probe.g_ky0 >= cx.g_ky0 && probe.g_kz0 >= cx.g_kz0 &&
          probe.g_kx0 + probe.g_nx <= cx.g_kx0 + cx.g_nx && probe.g_ky0 + probe.g_ny <= cx.g_ky0 + cx.g_ny &&
          probe.g_kz0 + probe.g_nz <= cx.g_kz0 + cx.g_nz)
        return KC_OK;
    } else {
      KC_TRY(fill_collision_window(c, x_lo, x_hi, y_lo, y_hi, probe, sz));
      if (probe.bm_kx0 >= cx.bm_kx0 && probe.bm_ky0 >= cx.bm_ky0 &&
          probe.bm_kx0 + probe.bm_cols <= cx.bm_kx0 + cx.bm_cols &&
          probe.bm_ky0 + probe.bm_rows <= cx.bm_ky0 + cx.bm_rows)
        return KC_OK;
    }
  }
  memset(&cx, 0, sizeof(cx));
  kc_planner_config c = h->cfg;
  c.octree_resolution = h->res_data;
  KC_TRY(fill_collision_frame(c, h->stw, h->sensor_tf_body, cx));
  Sizes sz;
  // grow the window so that neighbouring queries (a rollout, a planner's next samples) reuse it
  if (cx.coll_general) {
    const double pad = std::max(8.0 * cx.res, 0.25 * wreach);
    if (fill_collision_window_general(c, wcx, wcy, wreach + pad, cx, sz) != KC_OK)
      KC_TRY(fill_collision_window_general(c, wcx, wcy, wreach, cx, sz));
  } else {
    const double pad = std::max(32.0 * cx.res, 0.25 * std::max(x_hi - x_lo, y_hi - y_lo));
    if (fill_collision_window(c, x_lo - pad, x_hi + pad, y_lo - pad, y_hi + pad, cx, sz) != KC_OK)
      KC_TRY(fill_collision_window(c, x_lo, x_hi, y_lo, y_hi, cx, sz));
  }
  KC_REQUIRE(sz.sph_words <= ((size_t)1 << 27), KC_ERR_UNSUPPORTED,
             "sphere robot: voxel window of %d x %d columns is too large", cx.bm_cols, cx.bm_rows);
  cx.coll_enabled = h->n_sensor > 0 ? 1 : 0;
  cx.sensor_is_cloud = h->is_cloud;
  cx.n_sensor = h->n_sensor;
  cx.sensor = h->d_sensor.ptr;
  KC_TRY(h->d_bitmap.reserve(std::max<size_t>(sz.bitmap_words, 1)));
  cx.bitmap = h->d_bitmap.ptr;
  if (sz.sph_words) {
    KC_TRY(h->d_sph.reserve(sz.sph_words));
    cx.sph_col = h->d_sph.ptr;
  }
  KC_TRY(h->d_ctx.reserve(1));
  KC_CUDA(cudaMemcpyAsync(h->d_ctx.ptr, &cx, sizeof(cx), cudaMemcpyHostToDevice, h->stream));
  KC_CUDA(cudaMemsetAsync(h->d_bitmap.ptr, 0, std::max<size_t>(sz.bitmap_words, 1) * 4, h->stream));
  if (sz.sph_words)  // "no voxel in this column": +inf never passes the d2 <= r^2 test
    KC_CUDA(cudaMemsetAsync(h->d_sph.ptr, 0x7f, sz.sph_words * 4, h->stream));
  if (cx.coll_enabled) {
    const int gx = std::max(1, std::min((h->n_sensor + 255) / 256, 8 * sm_count()));
    k_prep_points<<<dim3(gx, 1), 256, 0, h->stream>>>(h->d_ctx.ptr);
    KC_CUDA(cudaGetLastError());
  }
  h->bitmap_valid = true;
  return KC_OK;
}

int32_t collision_set_sensor(kc_collision *h, const void *a, const void *b, int32_t n, bool cloud,
                             bool global_frame) {
  // ref: collision_check.h:99-101,121-125: sensor_tf_world_ is fixed at update time
  if (cloud && global_frame) {
    const float q[4] = {0, 0, 0, 1}, t[3] = {0, 0, 0};
    h->stw = hm::rigid_from_quat(q, t);
  } else {
    h->stw = hm::compose(hm::rigid_from_state(h->state[0], h->state[1], h->state[2]), h->sensor_tf_body);
  }
  h->res_data = h->cfg.octree_resolution;
  h->is_cloud = cloud ? 1 : 0;
  h->n_sensor = n;
  h->bitmap_valid = false;
  const size_t bytes = cloud ? (size_t)n * 12 : (size_t)n * 16;
  if (n > 0) {
    KC_TRY(h->d_sensor.reserve(bytes));
    KC_TRY(h->h_stage.reserve(bytes));
    if (cloud) {
      memcpy(h->h_stage.ptr, a, bytes);
    } else {
      memcpy(h->h_stage.ptr, a, (size_t)n * 8);
      memcpy(h->h_stage.ptr + (size_t)n * 8, b, (size_t)n * 8);
    }
    KC_CUDA(cudaMemcpyAsync(h->d_sensor.ptr, h->h_stage.ptr, bytes, cudaMemcpyHostToDevice, h->stream));
    KC_CUDA(cudaStreamSynchronize(h->stream));  // the staging buffer is reused by the next update
  }
  // surface an unsupported (tilted) mount at update time, like the DWA cycle does
  RobotCtx probe;
  memset(&probe, 0, sizeof(probe));
  return fill_collision_frame(h->cfg, h->stw, h->sensor_tf_body, probe);
}
}  // namespace

extern "C" {

int32_t kc_collision_create(const kc_collision_config *cfg, kc_collision **out) {
  KC_REQUIRE(out, KC_ERR_INVALID_ARG, "null output handle");
  *out = nullptr;
  KC_REQUIRE(cfg, KC_ERR_INVALID_ARG, "null config");
  KC_REQUIRE(cfg->robot_shape >= 0 && cfg->robot_shape <= 2, KC_ERR_INVALID_ARG,
             "Invalid robot geometry type");  // collision_check.cpp:56-58
  KC_REQUIRE(cfg->octree_resolution > 0.0, KC_ERR_OUT_OF_RANGE, "octree resolution must be positive");
  KC_TRY(ensure_device());
  kc_collision *h = new kc_collision();
  memset(&h->cfg, 0, sizeof(h->cfg));
  h->cfg.robot_shape = cfg->robot_shape;
  for (int i = 0; i < 3; ++i) h->cfg.robot_dims[i] = cfg->robot_dims[i];
  for (int i = 0; i < 3; ++i) h->cfg.sensor_position[i] = cfg->sensor_position[i];
  for (int i = 0; i < 4; ++i) h->cfg.sensor_rotation[i] = cfg->sensor_rotation[i];
  h->cfg.octree_resolution = cfg->octree_resolution;
  h->res_data = cfg->octree_resolution;
  h->sensor_tf_body = hm::rigid_from_quat(cfg->sensor_rotation, cfg->sensor_position);
  h->stw = h->sensor_tf_body;  // collision_check.cpp:67
  cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) {
    delete h;
    return cuda_fail(e, "stream creation", __FILE__, __LINE__);
  }
  *out = h;
  return KC_OK;
}

void kc_collision_destroy(kc_collision *h) {
  kc::ensure_device();  // the handle's device on this thread (frees below)
  if (!h) return;
  if (h->stream) cudaStreamSynchronize(h->stream);
  h->d_sensor.release();
  h->h_stage.release();
  h->d_bitmap.release();
  h->d_sph.release();
  h->d_states.release();
  h->d_out.release();
  h->d_ctx.release();
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

// ref: collision_check.cpp:70-75. Takes effect with the next sensor update (every user of the class
// updates the sensor data before checking).
int32_t kc_collision_reset_octree_resolution(kc_collision *h, double resolution) {
  KC_REQUIRE(h, KC_ERR_INVALID_ARG, "null handle");
  KC_REQUIRE(resolution > 0.0, KC_ERR_OUT_OF_RANGE, "octree resolution must be positive");
  KC_TRY(kc::ensure_device());
  h->cfg.octree_resolution = resolution;
  return KC_OK;
}

// ref: collision_check.cpp:39-55,77 getRadius
float kc_collision_get_radius(const kc_collision *h) {
  if (!h) return 0.0f;
  const double d0 = h->cfg.robot_dims[0], d1 = h->cfg.robot_dims[1];
  if (h->cfg.robot_shape == KC_BOX) return (float)(std::sqrt(d0 * d0 + d1 * d1) / 2);
  return (float)d0;
}

// ref: collision_check.cpp:125-147 updateState (both overloads)
int32_t kc_collision_update_state(kc_collision *h, double x, double y, double yaw) {
  KC_REQUIRE(h, KC_ERR_INVALID_ARG, "null handle");
  KC_TRY(kc::ensure_device());
  h->state[0] = x;
  h->state[1] = y;
  h->state[2] = yaw;
  return KC_OK;
}

// ref: collision_check.h:91-136 updateSensorData<LaserScan>
int32_t kc_collision_update_scan(kc_collision *h, const double *ranges, const double *angles, int32_t n) {
  KC_REQUIRE(h, KC_ERR_INVALID_ARG, "null handle");
  KC_REQUIRE(n >= 0 && (n == 0 || (ranges && angles)), KC_ERR_INVALID_ARG, "bad scan arrays");
  KC_TRY(kc::ensure_device());
  return collision_set_sensor(h, ranges, angles, n, false, false);
}

// ref: collision_check.h:91-136 updateSensorData<std::vector<Path::Point>>(data, global_frame)
int32_t kc_collision_update_cloud(kc_collision *h, const float *xyz, int32_t n, int32_t global_frame) {
  KC_REQUIRE(h, KC_ERR_INVALID_ARG, "null handle");
  KC_REQUIRE(n >= 0 && (n == 0 || xyz), KC_ERR_INVALID_ARG, "bad cloud");
  KC_TRY(kc::ensure_device());
  return collision_set_sensor(h, xyz, nullptr, n, true, global_frame != 0);
}

// ref: collision_check.cpp:225-246 checkCollisions(state), batched: collides[i] for states[i] =
// (x, y, yaw); *any = OR over the batch (TrajectorySampler::checkStatesFeasibility). Either output may
// be NULL.
int32_t kc_collision_check_states(kc_collision *h, const double *states, int32_t n, uint8_t *collides,
                                  int32_t *any) {
  KC_REQUIRE(h, KC_ERR_INVALID_ARG, "null handle");
  KC_REQUIRE(n >= 0 && (n == 0 || states), KC_ERR_INVALID_ARG, "bad state array");
  KC_TRY(kc::ensure_device());
  if (any) *any = 0;
  if (n == 0) return KC_OK;
  if (h->n_sensor == 0) {  // empty octree: nothing to hit
    if (collides) memset(collides, 0, (size_t)n);
    return KC_OK;
  }
  // octree-frame bounding box of the (finite) query positions, narrowed to float like the kernel
  const hm::Rot &L = h->stw.R;
  double x_lo = 1e300, x_hi = -1e300, y_lo = 1e300, y_hi = -1e300;
  double wx_lo = 1e300, wx_hi = -1e300, wy_lo = 1e300, wy_hi = -1e300;
  for (int32_t i = 0; i < n; ++i) {
    const double wx = (double)(float)states[3 * i], wy = (double)(float)states[3 * i + 1];
    const double dx = wx - (double)h->stw.t[0];
    const double dy = wy - (double)h->stw.t[1];
    const double px = (double)L(0, 0) * dx + (double)L(1, 0) * dy;
    const double py = (double)L(0, 1) * dx + (double)L(1, 1) * dy;
    if (!(std::abs(px) < 1e9 && std::abs(py) < 1e9 && std::abs(wx) < 1e9 && std::abs(wy) < 1e9)) continue;
    x_lo = std::min(x_lo, px);
    x_hi = std::max(x_hi, px);
    y_lo = std::min(y_lo, py);
    y_hi = std::max(y_hi, py);
    wx_lo = std::min(wx_lo, wx);
    wx_hi = std::max(wx_hi, wx);
    wy_lo = std::min(wy_lo, wy);
    wy_hi = std::max(wy_hi, wy);
  }
  if (x_lo > x_hi) {  // no finite pose: FCL reports no contact
    if (collides) memset(collides, 0, (size_t)n);
    return KC_OK;
  }
  KC_TRY(collision_prepare(h, x_lo, x_hi, y_lo, y_hi, wx_lo, wx_hi, wy_lo, wy_hi));
  KC_TRY(h->d_states.reserve((size_t)n * 3));
  KC_TRY(h->d_out.reserve((size_t)n + 8));
  KC_TRY(h->h_stage.reserve((size_t)n * 24 + (size_t)n + 16));
  memcpy(h->h_stage.ptr, states, (size_t)n * 24);
  KC_CUDA(cudaMemcpyAsync(h->d_states.ptr, h->h_stage.ptr, (size_t)n * 24, cudaMemcpyHostToDevice, h->stream));
  // flag word lives behind the per-state bytes (4-aligned)
  const size_t flag_off = ((size_t)n + 3) & ~(size_t)3;
  KC_CUDA(cudaMemsetAsync(h->d_out.ptr + flag_off, 0, 4, h->stream));
  const int gx = std::max(1, std::min((n + 127) / 128, 16 * sm_count()));
  (h->ctx.coll_general ? k_check_states<true> : k_check_states<false>)<<<gx, 128, 0, h->stream>>>(h->d_ctx.ptr, h->d_states.ptr, n, h->d_out.ptr,
                                            reinterpret_cast<int *>(h->d_out.ptr + flag_off));
  KC_CUDA(cudaGetLastError());
  uint8_t *hout = h->h_stage.ptr + (size_t)n * 24;
  KC_CUDA(cudaMemcpyAsync(hout, h->d_out.ptr, flag_off + 4, cudaMemcpyDeviceToHost, h->stream));
  KC_CUDA(cudaStreamSynchronize(h->stream));
  if (collides) memcpy(collides, hout, (size_t)n);
  if (any) {
    int32_t f;
    memcpy(&f, hout + flag_off, 4);
    *any = f != 0;
  }
  return KC_OK;
}

// ref: collision_check.cpp:149-162 checkCollisions() at the state set by updateState
int32_t kc_collision_check(kc_collision *h, int32_t *collides) {
  KC_REQUIRE(h && collides, KC_ERR_INVALID_ARG, "null argument");
  KC_TRY(kc::ensure_device());
  return kc_collision_check_states(h, h->state, 1, nullptr, collides);
}

}  // extern "C"
