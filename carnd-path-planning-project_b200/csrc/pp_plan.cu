// pp_plan.cu — the planning kernels and pp_plan_batch / pp_stats_batch.
//
// What bounds this path is FP64 instruction issue and branch divergence, not HBM
// (DESIGN.md §2: 1,520 algorithmic bytes against ~35 k FP64-heavy instructions
// per frame), and most of those instructions sit in serial recurrences.  So
// every LANE carries its own independent recurrence, and the step is cut into
// phases so that each phase runs with the mapping that keeps its lanes
// converged and its register / code footprint small:
//
//   k_prep     one thread per FRAME : ego state (src/main.cpp:1254-1282),
//              closest-waypoint scan + reference segment (:143-197), ego lane
//              matching + speed projection (:1302-1313)
//   k_cars     one thread per CAR   : Map::lane_matching + project_speed for
//              every sensor-fusion object (:1325-1350); warp tiles of 256 cars
//              counting-sorted by expected walk length
//   k_decide_t one thread per FRAME, tiles of 128 : LaneChangePlanner reductions,
//              veto, followed cars, LimitSpeed, SpeedController (:1352-1438),
//              TrajectoryBuilder set-up and the tk::spline fit (:565-904); the
//              tile's previous points come in by TMA bulk copies, the kept
//              points of the result leave by bulk stores from the same tile
//   k_emit     one thread per FRAME : the 0.02 s point emission loop
//              (:904-1040) on the <= 7 reachable knots staged in shared memory
//   k_fallback dense, side stream   : the angle-based generator (:848-901) for
//              the frames k_decide_t queued (~0.4 %)
//   k_slow     warp per frame, side : the complete path for frames k_emit gave
//              up on (headings / rotations outside its fast forms, ~0.03 %)
//
// The few hundred bytes per frame that cross between phases go through a
// double-buffered, stream-ordered scratch in HBM.  The ncu evidence behind each
// cut is in profiles/ (r1_v0: the single fused kernel, 45 % instruction-fetch
// stalls on 155 KB of SASS at 15 of 32 lanes; r1b/r1c: the division of the
// interior step at 4 lanes, the library atan2 at 3.6 lanes, knot staging; r2:
// the current state and the tile experiments of DESIGN.md §3.1).  Other forms of
// the same step, all bit-identical (tests/test_gpu_parity.py): variant 1, one
// thread per frame in one kernel (the cross-check); variant 3, k_cars_t (a
// warp's frames' cars by TMA into shared memory, reductions in the same kernel:
// half the DRAM traffic, 7 % slower); variant 4, plan_warp, one warp per frame
// (the default below 1,536 frames: 51 us for one frame).
#include <cuda.h>  // CUtensorMap (types only: the encoder is fetched through the runtime)
#include <cuda_runtime.h>

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "pp_device.cuh"
#include "pp_internal.h"

namespace {

using namespace ppd;

constexpr int kBlock = 128;
// minimum resident blocks per SM the compiler must allow for (register budget);
// tuned with ncu, see profiles/
// (profiles/sweep_minb.sh, gpurun_out/sweep2.log: prep 5 / cars 6 / decide 4 each gain 4-7 %;
// forcing the emission kernel below its natural 116 registers loses)
#ifndef PP_PREP_MINB
#define PP_PREP_MINB 5
#endif
#ifndef PP_CARS_MINB
#define PP_CARS_MINB 6
#endif
#ifndef PP_DECIDE_MINB
#define PP_DECIDE_MINB 4
#endif

// ---------------------------------------------------------------------------
// Stage A+B: ego state and reference segment (one frame).
// ---------------------------------------------------------------------------
struct FrameCtx {
  double x, y, speed, acc;  // ego pose / Cartesian speed / clamped acceleration
  int nprev;                // 0 or 10 kept points
  RefState rs;
  int lane;                 // ego lane (0 on match failure)
  double s, d, vs, vd;
  uint32_t flags;
};

// One point's term of the statistics' trajectory checksum (PP_STAT_XSUM, definition in
// include/pp.h): fixed point, 1/256 m, finite coordinates only.  Integer sums: order-free.
PPD_INLINE long long fx_point(double x, double y) {
  if (x == x && y == y && fabs(x) < 1e12 && fabs(y) < 1e12)
    return (long long)(x * 256.0) + (long long)(y * 256.0);
  return 0;
}
// add a thread's partial checksum to the global one: one atomic per warp (every lane calls)
PPD_INLINE void xsum_commit(unsigned long long *xsum, long long v) {
  unsigned long long u = (unsigned long long)v;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) u += __shfl_down_sync(0xffffffffu, u, o);
  if ((threadIdx.x & 31) == 0 && u) atomicAdd(xsum, u);
}
// a point sink that also accumulates the checksum of what passes through it
template <class Base>
struct SumOut {
  Base b;
  long long acc;
  PPD_INLINE void put(int i, double x, double y) {
    b.put(i, x, y);
    acc += fx_point(x, y);
  }
  PPD_INLINE void flush() { b.flush(); }
};

PPD_INLINE double ctx_dt0(const FrameCtx &c) { return c.nprev ? PP_PREV_KEEP / 50.0 : 0.0; }

// Ego state from the previous path or the telemetry (:1254-1282); (svx, svy) = speed vector.
PPD_INLINE void ego_state(const pp_frames &in, int64_t f, FrameCtx &c, double &svx, double &svy) {
  c.flags = 0;
  c.x = in.ego_x[f];
  c.y = in.ego_y[f];
  c.speed = in.ego_speed_mph[f];
  c.speed /= 2.237;  // :1239
  c.acc = 0;
  c.nprev = 0;
  svx = 0;
  svy = 0;
  if (in.prev_n[f] >= PP_PREV_KEEP) {  // :1261-1282
    const double *px = in.prev_x + f * PP_PREV_KEEP;
    const double *py = in.prev_y + f * PP_PREV_KEEP;
    const double p7x = px[7], p7y = py[7], p8x = px[8], p8y = py[8], p9x = px[9], p9y = py[9];
    const double v2 = vlen(p8x - p7x, p8y - p7y);
    svx = p9x - p8x;
    svy = p9y - p8y;
    const double v3 = vlen(svx, svy);
    c.acc = (v3 - v2) * 50;
    c.speed = v3 * 50;
    svx *= 50;
    svy *= 50;
    c.x = p9x;
    c.y = p9y;
    c.nprev = PP_PREV_KEEP;
  } else {
    c.flags |= PP_F_COLD_START;
  }
}

// Ego lane matching + speed projection (:1302-1320), given c.rs.
PPD_INLINE void ego_match(const MapView &m, const pp_config &cfg, FrameCtx &c, double svx,
                          double svy) {
  Match em = lane_match(m, c.rs, c.x, c.y);  // :1302-1307
  if (!em.ok) {
    c.flags |= PP_F_EGO_MATCH_FAIL;
    em.s = 0;
    em.d = 0;
    em.lane = 0;
  }
  c.lane = em.lane;
  c.s = em.s;
  c.d = em.d;
  project_speed(m, svx, svy, c.rs.wp, c.vs, c.vd);  // :1313
  if (c.acc > cfg.maximum_acc) c.acc = cfg.maximum_acc;  // :1319-1320
  if (c.acc < -cfg.maximum_acc) c.acc = -cfg.maximum_acc;
}

PPD_INLINE FrameCtx stage_prep(const MapView &m, const pp_config &cfg, const pp_frames &in,
                               int64_t f) {
  FrameCtx c;
  double svx, svy;
  ego_state(in, f, c, svx, svy);
  init_reference(m, c.x, c.y, c.rs);  // :1299
  ego_match(m, cfg, c, svx, svy);
  return c;
}

// ---------------------------------------------------------------------------
// Stage C: one sensor-fusion object (:1336-1343).
// ---------------------------------------------------------------------------
struct CarRes {
  int lane, wp;  // lane = -1: dropped (:1339)
  double s, d, vs, vd;
};

PPD_INLINE CarRes stage_car(const MapView &m, const RefState &rs, double x, double y, double vx,
                            double vy) {
  CarRes r;
  const Match cm = lane_match(m, rs, x, y);
  r.lane = cm.ok ? cm.lane : -1;
  r.wp = cm.ok ? cm.wp : 0;
  r.s = cm.s;
  r.d = cm.d;
  r.vs = 0;
  r.vd = 0;
  if (cm.ok) project_speed(m, vx, vy, cm.wp, r.vs, r.vd);
  return r;
}

// A slot of the car arrays: an ordinary car of the current message is matched (stage_car); a
// car the reference still holds from an earlier message (pp_frames::car_frozen_*) keeps the
// Frenet values of its last sighting (src/main.cpp:1194: nothing recomputes them).
PPD_INLINE CarRes car_slot(const MapView &m, const RefState &rs, const pp_frames &in, int64_t t,
                           double x, double y, double vx, double vy) {
  if (in.car_frozen_lane) {
    const int fl = in.car_frozen_lane[t];
    if (fl >= 0) {
      CarRes r;
      r.lane = fl;
      r.wp = 0;
      r.s = in.car_frozen_s[t];
      r.d = in.car_frozen_d[t];
      r.vs = in.car_frozen_vs[t];
      r.vd = in.car_frozen_vd[t];
      return r;
    }
  }
  return stage_car(m, rs, x, y, vx, vy);
}

// ---------------------------------------------------------------------------
// Stage D+E: streaming reductions over the cars of a frame
// (:377-445 LaneChangePlanner loop, :1388-1410 followed cars).
// ---------------------------------------------------------------------------
// Followed-car candidate: (s0, id) lexicographic minimum == the reference's
// "first car in ascending id order with strictly smaller s0" (:1395,1404).
struct Cand {
  double s0;
  int id, j;
};
PPD_INLINE void cand_init(Cand &c) {
  c.s0 = 0;
  c.id = -1;
  c.j = -1;
}
PPD_INLINE void cand_offer(Cand &c, double s0, int id, int j) {
  if (c.id == -1 || c.s0 > s0 || (c.s0 == s0 && id < c.id)) {
    c.s0 = s0;
    c.id = id;
    c.j = j;
  }
}

struct Behav {
  LaneStats ls;
  Cand own, tl0, tl1, tl2;
};
PPD_INLINE void behav_init(Behav &b, const pp_config &cfg) {
  lane_stats_init(b.ls, cfg);
  cand_init(b.own);
  cand_init(b.tl0);
  cand_init(b.tl1);
  cand_init(b.tl2);
}
// One matched car, given its predicted position (s0, d0) = (s + vs dt0, d + vd dt0) (:67-70).
PPD_INLINE void behav_add_pred(Behav &b, const pp_config &cfg, int ego_lane, double ego_s,
                               double ego_vs, double ego_d, int tl_in, int id, int j, int car_lane,
                               double s0, double car_vs, double d0, uint32_t &flags) {
  if (car_lane < 0) {  // :1336-1340 dropped from the map
    flags |= PP_F_CAR_DROPPED;
    return;
  }
  lane_stats_add_pred(b.ls, cfg, id, car_lane, s0, car_vs, ego_lane, tl_in, ego_s, ego_vs, flags);
  if (s0 > ego_s && fabs(d0 - ego_d) < 3) cand_offer(b.own, s0, id, j);
  if (s0 >= ego_s - cfg.car_length - cfg.safety_distance) {  // :1402
    if (fabs(d0 - lane_center_offset(0)) < 3) cand_offer(b.tl0, s0, id, j);
    if (fabs(d0 - lane_center_offset(1)) < 3) cand_offer(b.tl1, s0, id, j);
    if (fabs(d0 - lane_center_offset(2)) < 3) cand_offer(b.tl2, s0, id, j);
  }
}
PPD_INLINE void behav_add(Behav &b, const pp_config &cfg, const FrameCtx &c, int tl_in, int id,
                          int j, const CarRes &car, uint32_t &flags) {
  const double dt0 = ctx_dt0(c);
  behav_add_pred(b, cfg, c.lane, c.s, c.vs, c.d, tl_in, id, j, car.lane, car.s + car.vs * dt0,
                 car.vs, car.d + car.vd * dt0, flags);
}

// Every reduction of Behav is a lexicographic minimum, an AND or an OR, so partial results
// over disjoint sets of cars combine in any order: `b` += the partial result held by lane
// (own ^ mask); applied for every bit of a lane group this is a butterfly that leaves the
// group's total in each of its lanes (several lanes reduce one frame's cars, k_front).
PPD_INLINE void cand_merge_xor(Cand &c, int mask) {
  const double s0 = __shfl_xor_sync(0xffffffffu, c.s0, mask);
  const int id = __shfl_xor_sync(0xffffffffu, c.id, mask);
  const int j = __shfl_xor_sync(0xffffffffu, c.j, mask);
  if (id != -1) cand_offer(c, s0, id, j);
}
PPD_INLINE void behav_merge_xor(Behav &b, uint32_t &flags, int mask) {
#pragma unroll
  for (int l = 0; l < 3; l++) {
    const double os = __shfl_xor_sync(0xffffffffu, b.ls.next_s[l], mask);
    const int oid = __shfl_xor_sync(0xffffffffu, b.ls.next_id[l], mask);
    const double osp = __shfl_xor_sync(0xffffffffu, b.ls.speed[l], mask);
    // (a real entry always has s < 1000 = the default, so the default never wins a tie)
    const bool take = os < b.ls.next_s[l] || (os == b.ls.next_s[l] && oid < b.ls.next_id[l]);
    b.ls.next_s[l] = take ? os : b.ls.next_s[l];
    b.ls.next_id[l] = take ? oid : b.ls.next_id[l];
    b.ls.speed[l] = take ? osp : b.ls.speed[l];
  }
  b.ls.open &= __shfl_xor_sync(0xffffffffu, b.ls.open, mask);
  flags |= __shfl_xor_sync(0xffffffffu, flags, mask);
  cand_merge_xor(b.own, mask);
  cand_merge_xor(b.tl0, mask);
  cand_merge_xor(b.tl1, mask);
  cand_merge_xor(b.tl2, mask);
}

// ---------------------------------------------------------------------------
// Stage D..I tail: decision, speed target, trajectory, outputs (one frame).
// ---------------------------------------------------------------------------
struct Decision {
  int target_lane;
  SpeedCtl sc;
  uint32_t flags;
};

// lane decision, followed cars, speed target; writes every per-frame output
// except the trajectory itself, n_points and flags.
PPD_INLINE Decision stage_decide(const pp_config &cfg, const pp_frames &in, const pp_plans &out,
                                 int64_t f, const FrameCtx &c, const Behav &b, int tl_in,
                                 uint32_t flags) {
  const int64_t cb = f * in.max_cars;
  // lane decision (:1355) + veto (:1358-1369)
  int target_lane = lane_stats_decide(b.ls, cfg, c.lane, tl_in);
  if (target_lane != c.lane) {
    const double dtl = lane_center_offset(target_lane);
    const double diff = fabs(c.vd * 1.0 + c.d - dtl);
    if (diff > 6.0) {
      flags |= PP_F_VETO;
      target_lane = c.lane;
    }
  }
  Cand tl = target_lane == 0 ? b.tl0 : (target_lane == 1 ? b.tl1 : b.tl2);
  if (tl.id == b.own.id) tl.id = -1;  // :1411 only check once

  // speed target (:1422-1438)
  SpeedCtl sc;
  sc_init(sc, cfg, c.speed);
  if (b.own.id != -1) {
    double ts, tt;
    limit_speed(cfg, in.car_vx[cb + b.own.j], in.car_vy[cb + b.own.j], b.own.s0, c.s, c.speed,
                c.acc, true, ts, tt, flags);
    sc_limit(sc, ts, tt);
  }
  if (tl.id != -1) {
    double ts, tt;
    limit_speed(cfg, in.car_vx[cb + tl.j], in.car_vy[cb + tl.j], tl.s0, c.s, c.speed, c.acc, false,
                ts, tt, flags);
    sc_limit(sc, ts, tt);
  }
  if (out.target_speed) out.target_speed[f] = sc.target;
  if (out.target_time) out.target_time[f] = sc.time;
  out.ego_lane[f] = c.lane;
  out.ref_wp[f] = c.rs.wp;
  out.target_lane[f] = target_lane;
  if (out.ego_s) out.ego_s[f] = c.s;
  if (out.ego_d) out.ego_d[f] = c.d;
  if (out.ego_vs) out.ego_vs[f] = c.vs;
  if (out.ego_vd) out.ego_vd[f] = c.vd;
  if (out.ego_speed) out.ego_speed[f] = c.speed;
  if (out.ego_acc) out.ego_acc[f] = c.acc;
  if (out.next_car_id) out.next_car_id[f] = b.own.id;
  if (out.next_car_in_target_lane) out.next_car_in_target_lane[f] = tl.id;
  Decision d;
  d.target_lane = target_lane;
  d.sc = sc;
  d.flags = flags;
  return d;
}

PPD_INLINE void store_path_tail(const pp_plans &out, int64_t f, int np, uint32_t flags) {
  for (int i = np; i < PP_PATH_LEN; i++) {  // short (fallback) paths: pad with NaN
    out.next_x[f * PP_PATH_LEN + i] = __longlong_as_double(0x7ff8000000000000ll);
    out.next_y[f * PP_PATH_LEN + i] = __longlong_as_double(0x7ff8000000000000ll);
  }
  out.n_points[f] = np;
  out.flags[f] = flags;
}

// ---------------------------------------------------------------------------
// Stage D..I tail: decision, speed target, trajectory, outputs (one frame).
// ---------------------------------------------------------------------------
template <bool kLeanFirst = false>
PPD_INLINE void stage_finish(const MapView &m, const pp_config &cfg, const pp_frames &in,
                             const pp_plans &out, int64_t f, const FrameCtx &c, const Behav &b,
                             int tl_in, uint32_t flags0) {
  const Decision d = stage_decide(cfg, in, out, f, c, b, tl_in, flags0);
  uint32_t flags = d.flags;
  // trajectory (:1446-1448)
  const int np = build_trajectory<kLeanFirst>(m, cfg, c.rs, in.prev_x + f * PP_PREV_KEEP,
                                  in.prev_y + f * PP_PREV_KEEP, c.nprev, c.x, c.y,
                                  in.ego_yaw_deg[f], d.target_lane, c.d, c.vd, d.sc,
                                  out.next_x + f * PP_PATH_LEN, out.next_y + f * PP_PATH_LEN, flags);
  store_path_tail(out, f, np, flags);
}

PPD_INLINE void store_car(const pp_plans &out, int64_t slot, const CarRes &r) {
  if (out.car_lane) out.car_lane[slot] = r.lane;
  if (out.car_next_wp) out.car_next_wp[slot] = r.wp;
  if (out.car_s) out.car_s[slot] = r.s;
  if (out.car_d) out.car_d[slot] = r.d;
  if (out.car_vs) out.car_vs[slot] = r.vs;
  if (out.car_vd) out.car_vd[slot] = r.vd;
}

// The whole step for one frame, from its inputs alone.
PPD_INLINE void plan_one_frame(const MapView &m, const pp_config &cfg, const pp_frames &in,
                               const pp_plans &out, int64_t f) {
  const FrameCtx c = stage_prep(m, cfg, in, f);
  uint32_t flags = c.flags;
  const int mc = in.max_cars;
  int nc = in.n_cars[f];
  if (nc > mc) nc = mc;
  const int tl_in = in.target_lane_in[f];
  Behav b;
  behav_init(b, cfg);
  const int64_t cb = f * mc;
  for (int j = 0; j < nc; j++) {
    const CarRes r = car_slot(m, c.rs, in, cb + j, in.car_x[cb + j], in.car_y[cb + j],
                              in.car_vx[cb + j], in.car_vy[cb + j]);
    store_car(out, cb + j, r);
    behav_add(b, cfg, c, tl_in, in.car_id[cb + j], j, r, flags);
  }
  stage_finish(m, cfg, in, out, f, c, b, tl_in, flags);
}

// ===========================================================================
// Variant 4: one WARP per frame — the low-latency form for small batches (a single
// simulator's 50 Hz frames, a few hundred sessions in lockstep).  A frame's serial work cannot
// be cut (the emission loop is one recurrence, :908-1040), but everything that is a loop over
// independent items is spread over the 32 lanes: the closest-waypoint scan (:147-156) as six
// candidates per lane and a __shfl_xor argmin on (distance^2, index) — lowest index wins ties,
// like the reference's strict < in ascending order; the sensor-fusion loop (:1325-1350) with
// one lane per car; the reductions of LaneChangePlanner and the followed-car selection
// (:377-445, :1388-1410) as per-lane partial results merged by a shuffle butterfly.  The
// remaining serial phases run on all lanes redundantly (identical values, identical
// addresses): no divergence, no hand-over through memory, and a warp instruction costs the
// same for one active lane as for 32.
// ===========================================================================
PPD_INLINE int warp_closest_waypoint(const MapView &m, double x, double y) {
  const int lane = threadIdx.x & 31;
  int closest = lane < m.n ? lane : 0;
  double best = (m.t[closest * PP_MAP_STRIDE] - x) * (m.t[closest * PP_MAP_STRIDE] - x) +
                (m.t[closest * PP_MAP_STRIDE + 1] - y) * (m.t[closest * PP_MAP_STRIDE + 1] - y);
  for (int i = lane + 32; i < m.n; i += 32) {
    const double rx = m.t[i * PP_MAP_STRIDE], ry = m.t[i * PP_MAP_STRIDE + 1];
    const double d = (rx - x) * (rx - x) + (ry - y) * (ry - y);
    if (d < best) {
      closest = i;
      best = d;
    }
  }
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double od = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, closest, o);
    if (od < best || (od == best && oi < closest)) {
      best = od;
      closest = oi;
    }
  }
  // (every distance NaN: each lane kept its own first index; the reference answers 0)
  return __shfl_sync(0xffffffffu, closest, 0);
}

PPD_INLINE void plan_one_frame_warp(const MapView &m, const pp_config &cfg, const pp_frames &in,
                                    const pp_plans &out, int64_t f) {
  const int lane = threadIdx.x & 31;
  FrameCtx c;
  double svx, svy;
  ego_state(in, f, c, svx, svy);
  finish_reference(m, c.x, c.y, warp_closest_waypoint(m, c.x, c.y), c.rs);  // :1299
  ego_match(m, cfg, c, svx, svy);
  uint32_t flags = c.flags;
  const int mc = in.max_cars;
  int nc = in.n_cars[f];
  if (nc > mc) nc = mc;
  const int tl_in = in.target_lane_in[f];
  Behav b;
  behav_init(b, cfg);
  const int64_t cb = f * mc;
  for (int j = lane; j < nc; j += 32) {  // lane = car
    const CarRes r = car_slot(m, c.rs, in, cb + j, in.car_x[cb + j], in.car_y[cb + j],
                              in.car_vx[cb + j], in.car_vy[cb + j]);
    store_car(out, cb + j, r);
    behav_add(b, cfg, c, tl_in, in.car_id[cb + j], j, r, flags);
  }
  __syncwarp();
#pragma unroll 1
  for (int o = 1; o < 32; o <<= 1) behav_merge_xor(b, flags, o);
  stage_finish<true>(m, cfg, in, out, f, c, b, tl_in, flags);
}

__global__ void __launch_bounds__(kBlock)
plan_warp(const double *__restrict__ map_table, int n_wp, const __grid_constant__ pp_config cfg,
          const __grid_constant__ pp_frames in, const __grid_constant__ pp_plans out,
          int64_t n_frames) {
  extern __shared__ __align__(16) double s_map[];
  const MapView m = stage_map(s_map, map_table, n_wp);
  const int64_t warps = (int64_t)gridDim.x * (kBlock / 32);
  for (int64_t f = (int64_t)blockIdx.x * (kBlock / 32) + (threadIdx.x >> 5); f < n_frames; f += warps)
    plan_one_frame_warp(m, cfg, in, out, f);
}

// ===========================================================================
// Variant 1: everything in one kernel, one thread per frame.
// ===========================================================================
__global__ void __launch_bounds__(kBlock)
plan_fused(const double *__restrict__ map_table, int n_wp, const __grid_constant__ pp_config cfg,
           const __grid_constant__ pp_frames in, const __grid_constant__ pp_plans out,
           int64_t n_frames) {
  extern __shared__ __align__(16) double s_map[];
  const MapView m = stage_map(s_map, map_table, n_wp);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; f < n_frames; f += stride)
    plan_one_frame(m, cfg, in, out, f);
}

// ===========================================================================
// Variant 2: the three-phase pipeline.
// ===========================================================================
// Per-chunk scratch in HBM (SoA, one entry per frame / per car slot).
struct Scratch {
  double *x, *y, *speed, *acc, *s, *d, *vs, *vd, *ratio;  // ratio: [3][n]
  double *bh_d;   // tiled pipeline: the reduced Behav of every frame, [kBehavD][n]
  int32_t *bh_i;  // [kBehavI][n]
  int32_t *wp, *lane, *nprev;
  uint32_t *flags;
  double *car_s, *car_d, *car_vs, *car_vd;  // [n][max_cars]
  int32_t *car_lane;
  // between k_decide and k_emit: SpeedController, local frame, the reachable knots
  double *est;         // [kEstRows][n]
  int32_t *e_np;       // points already written (kept previous points)
  int32_t *e_nk;       // stored knots | kEstPartial; 0 = frame not for k_emit
  uint32_t *e_flags;   // flags raised so far
  // frames that need the complete path (k_slow): queue A is filled by k_decide, B by k_emit
  int32_t *slow_qa, *slow_qb;
  int32_t *slow_na, *slow_nb;
  int32_t *dbg;  // PP_DEBUG_SLOW: bail-out reasons of k_emit, else nullptr
  // pp_plan_stats_batch: the trajectory checksum is accumulated where the points are produced
  // (kept points in k_decide, new points in k_emit / k_fallback / k_slow) instead of re-reading
  // 800 B per frame afterwards; nullptr otherwise
  unsigned long long *xsum;
  int64_t n;  // frames in this chunk (stride of ratio)
};
constexpr int kEstHead = 7;  // sc.start, sc.target, sc.time, cx, cy, ca, sa
constexpr int kEstRows = kEstHead + 5 * PPD_TAILK;
constexpr int kEstPartial = 1 << 8;
constexpr int kEstFallback = 1 << 9;  // e_nk = kEstFallback | ncp: state for k_fallback, not k_emit

// The scratch of one chunk of n frames, carved by `cv` (see ppi::Carve).
Scratch carve_scratch(ppi::Carve &cv, int64_t n, int mc) {
  Scratch s = {};
  const size_t N = (size_t)n, NC = (size_t)n * (size_t)mc;
  cv.take(s.x, N);
  cv.take(s.y, N);
  cv.take(s.speed, N);
  cv.take(s.acc, N);
  cv.take(s.s, N);
  cv.take(s.d, N);
  cv.take(s.vs, N);
  cv.take(s.vd, N);
  cv.take(s.ratio, 3 * N);
  cv.take(s.wp, N);
  cv.take(s.lane, N);
  cv.take(s.nprev, N);
  cv.take(s.flags, N);
  cv.take(s.car_s, NC);
  cv.take(s.car_d, NC);
  cv.take(s.car_vs, NC);
  cv.take(s.car_vd, NC);
  cv.take(s.car_lane, NC);
  cv.take(s.est, (size_t)kEstRows * N);
  cv.take(s.e_np, N);
  cv.take(s.e_nk, N);
  cv.take(s.e_flags, N);
  // slow_qa / slow_qb / slow_na / slow_nb / dbg / xsum are set per chunk by the caller
  s.n = n;
  return s;
}

// Scratch of the tiled pipeline (variant 3): the ego context from k_prep (104 B per frame), the
// reduced Behav from k_cars_t (120 B), the emission state from k_decide_t.  The row stride is a
// multiple of 32 frames.
constexpr int kBehavDoubles = 10, kBehavInts = 10;
int64_t scratch3_stride(int64_t n) { return (n + 31) / 32 * 32; }
Scratch carve_scratch3(ppi::Carve &cv, int64_t n) {
  Scratch s = {};
  const size_t N = (size_t)scratch3_stride(n);
  cv.take(s.x, N);
  cv.take(s.y, N);
  cv.take(s.speed, N);
  cv.take(s.acc, N);
  cv.take(s.s, N);
  cv.take(s.d, N);
  cv.take(s.vs, N);
  cv.take(s.vd, N);
  cv.take(s.ratio, 3 * N);
  cv.take(s.wp, N);
  cv.take(s.lane, N);
  cv.take(s.nprev, N);
  cv.take(s.flags, N);
  cv.take(s.bh_d, (size_t)kBehavDoubles * N);
  cv.take(s.bh_i, (size_t)kBehavInts * N);
  cv.take(s.est, (size_t)kEstRows * N);
  cv.take(s.e_np, N);
  cv.take(s.e_nk, N);
  cv.take(s.e_flags, N);
  s.n = (int64_t)N;
  return s;
}

// One chunk's scratch at `base` (variant 3: the tiled pipeline's); a null base only sizes it.
Scratch carve_chunk(char *base, bool tiled, int64_t n, int mc, size_t *bytes = nullptr) {
  ppi::Carve cv(base);
  const Scratch s = tiled ? carve_scratch3(cv, n) : carve_scratch(cv, n, mc);
  if (bytes) *bytes = cv.size;
  return s;
}

// `in` / `out` already point at the first frame of the chunk.
__global__ void __launch_bounds__(kBlock, PP_PREP_MINB)
k_prep(const double *__restrict__ map_table, int n_wp, const __grid_constant__ pp_config cfg,
       const __grid_constant__ pp_frames in, const __grid_constant__ Scratch sc, int64_t n) {
  extern __shared__ __align__(16) double s_map[];
  const MapView m = stage_map(s_map, map_table, n_wp);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; f < n; f += stride) {
    const FrameCtx c = stage_prep(m, cfg, in, f);
    sc.x[f] = c.x;
    sc.y[f] = c.y;
    sc.speed[f] = c.speed;
    sc.acc[f] = c.acc;
    sc.s[f] = c.s;
    sc.d[f] = c.d;
    sc.vs[f] = c.vs;
    sc.vd[f] = c.vd;
    sc.ratio[f] = c.rs.ratio[0];
    sc.ratio[sc.n + f] = c.rs.ratio[1];
    sc.ratio[2 * sc.n + f] = c.rs.ratio[2];
    sc.wp[f] = c.rs.wp;
    sc.lane[f] = c.lane;
    sc.nprev[f] = c.nprev;
    sc.flags[f] = c.flags;
  }
}

// One thread per car.  The number of segments a car's walk takes grows with its
// distance from the ego along the road, and a warp advances at the pace of its
// longest walk (ncu, profiles/r1c: 75 % of this kernel's instructions were in
// the walk loop at 13 of 32 lanes).  So each warp takes a tile of 32 x kTileK
// consecutive car slots, bins them by a cheap proxy of the walk length
// (distance to the ego in units of the local segment length), counting-sorts
// the tile in shared memory and then walks 32 cars of similar length at a time.
// The proxy only orders the work; results do not depend on it.
#ifndef PP_TILE_K
#define PP_TILE_K 8
#endif
// kTileK = cars per lane per tile (a tile is 32 kTileK car slots).  8 is the throughput setting
// (profiles/r2_tilek.log: 4 -> 1.01 ms, 8 -> 0.97, 16 -> 1.21 per 1M frames); a chunk too small to
// give every resident warp a tile of 256 takes tiles of 64, which spreads it over four times as
// many warps and quarters the kernel's latency (closed-loop rollouts tick in chunks of 8,192
// frames: their chain of dependent launches is what bounds them).
constexpr int kTileKBig = PP_TILE_K, kTileKSmall = 2;
constexpr int kBins = 24;              // proxy bins; bin kBins = slot holds no car
template <int kTileK>
__global__ void __launch_bounds__(kBlock, PP_CARS_MINB)
k_cars(const double *__restrict__ map_table, int n_wp, const __grid_constant__ pp_frames in,
       const __grid_constant__ pp_plans out, const __grid_constant__ Scratch sc, int64_t n) {
  constexpr int kTile = 32 * kTileK;  // car slots per tile
  extern __shared__ __align__(16) double s_map[];
  __shared__ int s_hist[kBlock / 32][32];
  __shared__ unsigned short s_order[kBlock / 32][kTile];
  const MapView m = stage_map(s_map, map_table, n_wp);
  const int mc = in.max_cars;
  const unsigned mc_magic = mc > 0 ? 0xFFFFFFFFu / (unsigned)mc + 1u : 0u;  // exact below 2^32 / mc
  const int64_t total = n * mc;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  int *hist = s_hist[wib];
  unsigned short *order = s_order[wib];
  const int64_t n_tiles = (total + kTile - 1) / kTile;
  const int64_t warps = (int64_t)gridDim.x * (kBlock / 32);
  for (int64_t tile = (int64_t)blockIdx.x * (kBlock / 32) + wib; tile < n_tiles; tile += warps) {
    const int64_t base = tile * kTile;
    // frame and slot of item base + i are f0 + (r0 + i) / mc and (r0 + i) % mc; r0 + i is small,
    // so one multiply-high by mc_magic = ceil(2^32 / mc) divides it exactly (the 64-bit division
    // per item this replaces was ~5 % of the kernel's instructions)
    const int64_t f0 = base / mc;
    const unsigned r0 = (unsigned)(base - f0 * mc);
    // ---- bin the tile's cars
    hist[lane] = 0;
    __syncwarp();
    int key[kTileK];  // bin | rank within the bin << 8
    // pass 1: the bins.  Every load is unconditional (slots past n_cars are allocated padding,
    // a clamped index keeps the last tile in range) and independent of the others, so the
    // loads of all eight items go out together; as `if (j < n_cars[f]) { load ... }` each item
    // cost two dependent trips to memory.
#pragma unroll
    for (int k = 0; k < kTileK; k++) {
      const int64_t t = base + k * 32 + lane;
      const bool in_range = t < total;
      const int64_t tc = in_range ? t : total - 1;
      const unsigned xi = r0 + (unsigned)(tc - base);
      const unsigned qi = mc == 1 ? xi : __umulhi(xi, mc_magic);  // (the magic wraps to 0 for 1)
      const int64_t f = f0 + qi;
      const int j = (int)(xi - qi * (unsigned)mc);
      const int nc = in.n_cars[f];
      const float dx = (float)(in.car_x[tc] - sc.x[f]), dy = (float)(in.car_y[tc] - sc.y[f]);
      const int wp = sc.wp[f];
      const float len = (float)row(m, wp)[11];  // centre lane's segment length
      const float q = sqrtf(dx * dx + dy * dy) / len;
      const int b = q < (float)(kBins - 1) ? (int)q : kBins - 1;  // NaN -> last bin
      key[k] = (in_range & (j < nc)) ? b : kBins;
    }
    // pass 2: rank within the bin
#pragma unroll
    for (int k = 0; k < kTileK; k++) key[k] |= atomicAdd(&hist[key[k]], 1) << 8;
    __syncwarp();
    // exclusive prefix over the bins (lane b owns bin b)
    const int cnt = hist[lane];
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    __syncwarp();
    hist[lane] = incl - cnt;
    __syncwarp();
    const int n_valid = hist[kBins];
#pragma unroll
    for (int k = 0; k < kTileK; k++)
      order[hist[key[k] & 0xff] + (key[k] >> 8)] = (unsigned short)(k * 32 + lane);
    __syncwarp();
    // ---- walk them, 32 of similar length at a time
    for (int g = lane; g < n_valid; g += 32) {
      const unsigned oi = order[g];
      const int64_t t = base + oi;
      const unsigned qi = mc == 1 ? r0 + oi : __umulhi(r0 + oi, mc_magic);
      const int64_t f = f0 + qi;
      const int j = (int)(r0 + oi - qi * (unsigned)mc);
      RefState rs;
      rs.wp = sc.wp[f];
      rs.ratio[0] = sc.ratio[f];
      rs.ratio[1] = sc.ratio[sc.n + f];
      rs.ratio[2] = sc.ratio[2 * sc.n + f];
      const CarRes r = car_slot(m, rs, in, t, in.car_x[t], in.car_y[t], in.car_vx[t], in.car_vy[t]);
      const int64_t slot = (int64_t)j * sc.n + f;  // car-major: k_decide reads it coalesced
      sc.car_s[slot] = r.s;
      sc.car_d[slot] = r.d;
      sc.car_vs[slot] = r.vs;
      sc.car_vd[slot] = r.vd;
      sc.car_lane[slot] = r.lane;
      store_car(out, t, r);
    }
    __syncwarp();
  }
}

// Everything of a frame after the per-car phase, from the scratch of k_prep /
// k_cars: the complete path (any frame).
PPD_INLINE void load_ctx(const Scratch &sc, int64_t f, FrameCtx &c) {
  c.x = sc.x[f];
  c.y = sc.y[f];
  c.speed = sc.speed[f];
  c.acc = sc.acc[f];
  c.s = sc.s[f];
  c.d = sc.d[f];
  c.vs = sc.vs[f];
  c.vd = sc.vd[f];
  c.rs.ratio[0] = sc.ratio[f];
  c.rs.ratio[1] = sc.ratio[sc.n + f];
  c.rs.ratio[2] = sc.ratio[2 * sc.n + f];
  c.rs.wp = sc.wp[f];
  c.lane = sc.lane[f];
  c.nprev = sc.nprev[f];
  c.flags = sc.flags[f];
}
PPD_INLINE void reduce_cars(const pp_config &cfg, const pp_frames &in, const Scratch &sc, int64_t f,
                            const FrameCtx &c, int tl_in, Behav &b, uint32_t &flags) {
  const int mc = in.max_cars;
  int nc = in.n_cars[f];
  if (nc > mc) nc = mc;
  behav_init(b, cfg);
  const int64_t cb = f * mc;
  // car j + 1 is loaded while car j is reduced (the loads are coalesced: car-major scratch)
  CarRes nxt;
  int nxt_id = 0;
  auto fetch = [&](int j) {
    const int64_t slot = (int64_t)j * sc.n + f;
    nxt.lane = sc.car_lane[slot];
    nxt.wp = 0;
    nxt.s = sc.car_s[slot];
    nxt.d = sc.car_d[slot];
    nxt.vs = sc.car_vs[slot];
    nxt.vd = sc.car_vd[slot];
    nxt_id = in.car_id[cb + j];
  };
  if (nc > 0) fetch(0);
  for (int j = 0; j < nc; j++) {
    const CarRes r = nxt;
    const int id = nxt_id;
    if (j + 1 < nc) fetch(j + 1);
    behav_add(b, cfg, c, tl_in, id, j, r, flags);
  }
}

template <class S>
PPD_INLINE S make_sink(double *x, double *y);
template <>
PPD_INLINE ArrayOut make_sink<ArrayOut>(double *x, double *y) {
  return ArrayOut{x, y};
}
template <>
PPD_INLINE PairOut make_sink<PairOut>(double *x, double *y) {
  return PairOut{x, y, 0.0, 0.0, -1};
}

// The emission loop (one thread per frame): no map, no spline fit, no library
// transcendental — small code, few registers, many resident warps.  The
// reachable knots are staged in shared memory (one column per thread).  A frame
// that leaves the ranges the fast forms cover re-plans through k_slow.
#ifndef PP_EMIT_MINB
#define PP_EMIT_MINB 4
#endif
// PointSink: PairOut when next_x / next_y are 16-byte aligned, else ArrayOut; kSum: also
// accumulate the statistics' checksum (sc.xsum)
template <class PointSink, bool kSum>
__global__ void __launch_bounds__(kBlock, PP_EMIT_MINB)
k_emit(const __grid_constant__ pp_config cfg, const __grid_constant__ pp_plans out,
       const __grid_constant__ Scratch sc, int64_t n) {
  extern __shared__ double s_knots[];  // [5 * PPD_TAILK][blockDim.x]
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  long long xacc = 0;  // checksum of the points emitted here (frames that bail out add nothing)
  for (int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; f < n; f += stride) {
    const int code = sc.e_nk[f];
    if (code & kEstFallback) continue;  // queued for k_fallback
    const int cnt = code & (kEstPartial - 1);
    const double *e = sc.est + f;
    SpeedCtl ctl;
    ctl.shift = 0;
    ctl.start = e[0 * sc.n];
    ctl.target = e[1 * sc.n];
    ctl.time = e[2 * sc.n];
    const double cx = e[3 * sc.n], cy = e[4 * sc.n], ca = e[5 * sc.n], sa = e[6 * sc.n];
    double *col = s_knots + threadIdx.x;
    // all 35 slots, unconditionally: fixed trip counts let the loads of a row go out
    // together (slots past cnt hold stale values that are never read)
#pragma unroll
    for (int r = 0; r < 5; r++) {
      double tmp[PPD_TAILK];
#pragma unroll
      for (int k = 0; k < PPD_TAILK; k++) tmp[k] = e[(kEstHead + r * PPD_TAILK + k) * sc.n];
#pragma unroll
      for (int k = 0; k < PPD_TAILK; k++) col[(r * PPD_TAILK + k) * blockDim.x] = tmp[k];
    }
    KnotsTail kn;
    kn.base = col;
    kn.stride = blockDim.x;
    kn.count = cnt;
    kn.part = (code & kEstPartial) != 0;
    uint32_t flags = sc.e_flags[f];
    int bail;
    int np;
    if (kSum) {
      SumOut<PointSink> pts{make_sink<PointSink>(out.next_x + f * PP_PATH_LEN,
                                                 out.next_y + f * PP_PATH_LEN), 0};
      np = traj_emit_lean(kn, cfg, ctl, cx, cy, ca, sa, sc.e_np[f], pts, flags, bail);
      if (!bail) xacc += pts.acc;
    } else {
      PointSink pts = make_sink<PointSink>(out.next_x + f * PP_PATH_LEN, out.next_y + f * PP_PATH_LEN);
      np = traj_emit_lean(kn, cfg, ctl, cx, cy, ca, sa, sc.e_np[f], pts, flags, bail);
    }
    if (bail) {
      sc.slow_qb[atomicAdd(sc.slow_nb, 1)] = (int32_t)f;
      if (sc.dbg) atomicAdd(sc.dbg + bail, 1);
      continue;
    }
    store_path_tail(out, f, np, flags);
  }
  if (kSum) xsum_commit(sc.xsum, xacc);
}

// The angle-based generator (:848-901) for the frames k_decide queued.  Every
// lane runs the same loop, so the queue is consumed densely (32 frames a warp).
__global__ void __launch_bounds__(kBlock)
k_fallback(const __grid_constant__ pp_plans out, const __grid_constant__ Scratch sc,
           const int32_t *__restrict__ queue, const int32_t *__restrict__ queue_n) {
  const int count = *queue_n;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  long long xacc = 0;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < count; q += stride) {
    const int64_t f = queue[q];
    const double *e = sc.est + f;
    SpeedCtl ctl;
    ctl.shift = 0;
    ctl.start = e[0 * sc.n];
    ctl.target = e[1 * sc.n];
    ctl.time = e[2 * sc.n];
    TrajFrame tf;
    tf.cx = e[3 * sc.n];
    tf.cy = e[4 * sc.n];
    tf.ca = e[5 * sc.n];
    tf.sa = e[6 * sc.n];
#pragma unroll
    for (int k = 0; k < 6; k++) {
      tf.cpx[k] = e[(kEstHead + k) * sc.n];
      tf.cpy[k] = e[(kEstHead + 6 + k) * sc.n];
    }
    tf.np = sc.e_np[f];
    tf.ncp = sc.e_nk[f] & 0xff;
    const int np = traj_fallback(tf, ctl, out.next_x + f * PP_PATH_LEN, out.next_y + f * PP_PATH_LEN);
    store_path_tail(out, f, np, sc.e_flags[f]);
    if (sc.xsum)  // the new points (the kept ones were counted by k_decide)
      for (int i = tf.np; i < np; i++)
        xacc += fx_point(out.next_x[f * PP_PATH_LEN + i], out.next_y[f * PP_PATH_LEN + i]);
  }
  if (sc.xsum) xsum_commit(sc.xsum, xacc);
}

// The complete path for the frames k_emit gave up on (a few hundred per
// million: headings or frame rotations outside the ranges its fast forms
// cover, arguments left of the staged knots).  Every such frame takes its own
// route through the code, so each gets a warp of its own (lane 0): nothing is
// serialised behind another frame's branches.
constexpr int kSlowSpread = 32;
__global__ void __launch_bounds__(kBlock)
k_slow(const double *__restrict__ map_table, int n_wp, const __grid_constant__ pp_config cfg,
       const __grid_constant__ pp_frames in, const __grid_constant__ pp_plans out,
       const __grid_constant__ Scratch sc, const int32_t *__restrict__ queue,
       const int32_t *__restrict__ queue_n) {
  const int count = *queue_n;
  const int per_block = kBlock / kSlowSpread;
  if ((int64_t)blockIdx.x * per_block >= count) return;
  extern __shared__ __align__(16) double s_map[];
  const MapView m = stage_map(s_map, map_table, n_wp);
  if (threadIdx.x % kSlowSpread) return;
  const int64_t stride = (int64_t)gridDim.x * per_block;
  for (int64_t q = (int64_t)blockIdx.x * per_block + threadIdx.x / kSlowSpread; q < count;
       q += stride) {
    const int64_t f = queue[q];
    FrameCtx c;
    load_ctx(sc, f, c);
    uint32_t flags = c.flags;
    const int tl_in = in.target_lane_in[f];
    Behav b;
    reduce_cars(cfg, in, sc, f, c, tl_in, b, flags);
    stage_finish(m, cfg, in, out, f, c, b, tl_in, flags);
    if (sc.xsum) {  // new points of the re-planned frame (rare: one atomic per frame is fine)
      long long xacc = 0;
      const int np = out.n_points[f];
      for (int i = c.nprev; i < np; i++)
        xacc += fx_point(out.next_x[f * PP_PATH_LEN + i], out.next_y[f * PP_PATH_LEN + i]);
      if (xacc) atomicAdd(sc.xsum, (unsigned long long)xacc);
    }
  }
}

// ===========================================================================
// Variant 3: the tiled pipeline.  Same phases as variant 2, but a frame TILE is the unit of
// memory traffic where that pays: the cars of a warp's frames arrive in shared memory by TMA
// bulk copies and their results never leave the SM (the reductions of LaneChangePlanner and
// the followed-car selection run in the kernel that matched the cars: 120 B per frame go on
// instead of 36 B per car written and read back), and the decision kernel gets the previous
// points of its 128 frames by one bulk copy per coordinate and copies the kept points out of
// the same tile.
//
//   k_prep     (as variant 2) one thread per frame
//   k_cars_t   one WARP per tile of F = min(32, 256 / max_cars) consecutive frames: the
//              tile's cars bulk-copied into shared memory, counting-sorted by expected walk
//              length and matched (lane = car), results written over the inputs in place;
//              then the per-frame reductions (:377-445, :1388-1410; G lanes per frame,
//              merged with a shuffle butterfly when traffic is dense)
//   k_decide_t one thread per frame, tiles of 128: lane decision, veto, followed cars,
//              LimitSpeed, SpeedController (:1355-1438), TrajectoryBuilder set-up and the
//              tk::spline fit (:565-904)
//   k_emit     (as variant 2)
//
// Measured and dropped (profiles/r2_probe_*.log): one fused front kernel (ego state + cars +
// reductions + decision; the state it carries across the car phase spills, 1.82 ms against
// 1.49 ms for the separate kernels), knot rows by TMA into the emission kernel (0.92 against
// 0.87 ms: a block-synchronous tile loop exposes the slowest lane and the load latency once
// per tile) and per-lane 80-byte bulk stores of the emitted points (1.01 ms: a bulk copy is
// issued lane by lane, 64 of them replace 10 vector stores).
// ===========================================================================
struct CarsGeom {
  int F;        // frames per warp tile
  int G;        // lanes per frame in the reduction (power of two, F * G <= 32)
  int T;        // car slots per tile (F * max_cars rounded up to even)
  int Cg;       // max_cars rounded up to a multiple of G
  int warp_bytes;  // shared memory per warp
  unsigned magic;  // ceil(2^16 / max_cars): i / max_cars for i < 256
  int bulk;     // car arrays are 16-byte aligned: tiles come by TMA
};

// per-warp shared memory: car[4][T] doubles | 8 per-frame double arrays [Fc] | 5 per-frame int
// arrays [Fc] | hist[32] ints | order[256] bytes | mbarrier     (Fc = F rounded up to even)
__host__ __device__ inline int cars_warp_bytes(int T, int F) {
  const int Fc = (F + 1) & ~1;
  const int b = 4 * T * 8 + 8 * Fc * 8 + 5 * Fc * 4 + 32 * 4 + 256 + 16;
  return (b + 15) & ~15;
}
// what a matched car contributes to its frame's reductions, packed next to its lane
constexpr unsigned kFactCloses = 1u << 31;  // closes its lane (:405-444)
constexpr unsigned kFactOwn = 1u << 27;     // ahead in the ego's corridor (:1388-1398)
constexpr unsigned kFactTl0 = 1u << 28;     // candidate for target lane 0 / 1 / 2 (:1402-1410)
constexpr unsigned kFactFlags = PP_F_CLOSED_RANGE | PP_F_CLOSED_AHEAD | PP_F_CLOSED_BEHIND;
static_assert((kFactFlags & (kFactCloses | (15u << 27))) == 0, "fact bits overlap the flags");

constexpr int kCarRounds = 8;  // 32-item rounds per tile (<= 256 car slots)
static_assert(kBehavDoubles == 10 && kBehavInts == 10, "behav_store / behav_load layout");

PPD_INLINE void behav_store(const Scratch &sc, int64_t f, const Behav &b, uint32_t flags) {
  double *d = sc.bh_d + f;
  int32_t *i = sc.bh_i + f;
  const int64_t n = sc.n;
#pragma unroll
  for (int l = 0; l < 3; l++) {
    d[l * n] = b.ls.next_s[l];
    d[(3 + l) * n] = b.ls.speed[l];
  }
  d[6 * n] = b.own.s0;
  d[7 * n] = b.tl0.s0;
  d[8 * n] = b.tl1.s0;
  d[9 * n] = b.tl2.s0;
  i[0 * n] = (int32_t)b.ls.open;
  i[1 * n] = (int32_t)flags;
  i[2 * n] = b.own.id;
  i[3 * n] = b.own.j;
  i[4 * n] = b.tl0.id;
  i[5 * n] = b.tl0.j;
  i[6 * n] = b.tl1.id;
  i[7 * n] = b.tl1.j;
  i[8 * n] = b.tl2.id;
  i[9 * n] = b.tl2.j;
}
PPD_INLINE void behav_load(const Scratch &sc, const pp_config &cfg, int64_t f, Behav &b,
                           uint32_t &flags) {
  const double *d = sc.bh_d + f;
  const int32_t *i = sc.bh_i + f;
  const int64_t n = sc.n;
  behav_init(b, cfg);
#pragma unroll
  for (int l = 0; l < 3; l++) {
    b.ls.next_s[l] = d[l * n];
    b.ls.speed[l] = d[(3 + l) * n];
  }
  b.own.s0 = d[6 * n];
  b.tl0.s0 = d[7 * n];
  b.tl1.s0 = d[8 * n];
  b.tl2.s0 = d[9 * n];
  b.ls.open = (unsigned)i[0 * n];
  flags |= (uint32_t)i[1 * n];
  b.own.id = i[2 * n];
  b.own.j = i[3 * n];
  b.tl0.id = i[4 * n];
  b.tl0.j = i[5 * n];
  b.tl1.id = i[6 * n];
  b.tl1.j = i[7 * n];
  b.tl2.id = i[8 * n];
  b.tl2.j = i[9 * n];
}

template <int kThreads>
__global__ void __launch_bounds__(kThreads, 1)
k_cars_t(const double *__restrict__ map_table, int n_wp, const __grid_constant__ pp_config cfg,
         const __grid_constant__ pp_frames in, const __grid_constant__ pp_plans out,
         const __grid_constant__ Scratch sc, int64_t n, const __grid_constant__ CarsGeom g) {
  extern __shared__ __align__(16) double s_dyn[];
  const MapView m = stage_map(s_dyn, map_table, n_wp);
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  char *wbase = reinterpret_cast<char *>(s_dyn) + map_stage_bytes(n_wp) + (size_t)wib * g.warp_bytes;
  double *car0 = reinterpret_cast<double *>(wbase);  // x -> predicted s
  double *car1 = car0 + g.T;                          // y -> predicted d
  double *car2 = car1 + g.T;                          // vx -> vs
  double *car3 = car2 + g.T;                          // vy -> lane (int)
  const int Fc = (g.F + 1) & ~1;
  double *fx = car3 + g.T, *fy = fx + Fc, *fr0 = fy + Fc, *fr1 = fr0 + Fc, *fr2 = fr1 + Fc;
  double *fes = fr2 + Fc, *fevs = fes + Fc, *fed = fevs + Fc;  // ego s, vs, d
  int *fwp = reinterpret_cast<int *>(fed + Fc), *fnc = fwp + Fc, *fnp = fnc + Fc;
  int *fel = fnp + Fc, *ftl = fel + Fc;  // ego lane, incoming target lane
  int *hist = ftl + Fc;
  unsigned char *order = reinterpret_cast<unsigned char *>(hist + 32);
  unsigned long long *bar_p = reinterpret_cast<unsigned long long *>(
      (reinterpret_cast<uintptr_t>(order + 256) + 7) & ~(uintptr_t)7);
  const unsigned bar = smem_addr(bar_p);
  if (lane == 0) mbar_init(bar, 1);
  __syncwarp();
  const int mc = in.max_cars, F = g.F, G = g.G;
  const Rcp racc = rcp_make(cfg.relaxed_acc);
  const int64_t n_tiles = (n + F - 1) / F;
  const int64_t warps = (int64_t)gridDim.x * (kThreads / 32);
  unsigned phase = 0;
  for (int64_t tile = (int64_t)blockIdx.x * (kThreads / 32) + wib; tile < n_tiles; tile += warps) {
    const int64_t f0 = tile * F;
    const int nf = (int)((n - f0) < F ? (n - f0) : F);
    const int items = nf * mc;
    const int64_t cb0 = f0 * mc;
    // ---- the tile's cars: one bulk copy per array (ordinary loads when unaligned)
    const bool bulk = g.bulk && !(items & 1);
    if (bulk) {
      if (lane == 0) {
        const unsigned bytes = (unsigned)items * 8u;
        mbar_expect_tx(bar, 4u * bytes);
        bulk_g2s(smem_addr(car0), in.car_x + cb0, bytes, bar);
        bulk_g2s(smem_addr(car1), in.car_y + cb0, bytes, bar);
        bulk_g2s(smem_addr(car2), in.car_vx + cb0, bytes, bar);
        bulk_g2s(smem_addr(car3), in.car_vy + cb0, bytes, bar);
      }
    } else {
      for (int i = lane; i < items; i += 32) {
        car0[i] = in.car_x[cb0 + i];
        car1[i] = in.car_y[cb0 + i];
        car2[i] = in.car_vx[cb0 + i];
        car3[i] = in.car_vy[cb0 + i];
      }
    }
    // ---- what the car lanes need of their frames (lane = frame here)
    if (lane < nf) {
      const int64_t f = f0 + lane;
      fx[lane] = sc.x[f];
      fy[lane] = sc.y[f];
      fr0[lane] = sc.ratio[f];
      fr1[lane] = sc.ratio[sc.n + f];
      fr2[lane] = sc.ratio[2 * sc.n + f];
      fwp[lane] = sc.wp[f];
      const int nc = in.n_cars[f];
      fnc[lane] = nc > mc ? mc : nc;
      fnp[lane] = sc.nprev[f];
      fes[lane] = sc.s[f];
      fevs[lane] = sc.vs[f];
      fed[lane] = sc.d[f];
      fel[lane] = sc.lane[f];
      ftl[lane] = in.target_lane_in[f];
    }
    hist[lane] = 0;
    __syncwarp();
    if (bulk) {
      mbar_wait(bar, phase);
      phase ^= 1;
    }
    // ---- bin the cars by expected walk length (distance to the ego in units of the local
    // segment length); the proxy only orders the work
    int key[kCarRounds];
#pragma unroll
    for (int k = 0; k < kCarRounds; k++) {
      key[k] = kBins;
      if (k * 32 < items) {
        const int i = k * 32 + lane;
        const int ic = i < items ? i : items - 1;
        const int fl = (int)(((unsigned)ic * g.magic) >> 16);
        const int j = ic - fl * mc;
        const float dx = (float)(car0[ic] - fx[fl]), dy = (float)(car1[ic] - fy[fl]);
        const float len = (float)row(m, fwp[fl])[11];  // centre lane's segment length
        const float q = sqrtf(dx * dx + dy * dy) / len;
        const int bin = q < (float)(kBins - 1) ? (int)q : kBins - 1;  // NaN -> last bin
        key[k] = ((i < items) & (j < fnc[fl])) ? bin : kBins;
      }
    }
#pragma unroll
    for (int k = 0; k < kCarRounds; k++)
      if (k * 32 < items) key[k] |= atomicAdd(&hist[key[k]], 1) << 8;
    __syncwarp();
    const int cnt = hist[lane];
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    __syncwarp();
    hist[lane] = incl - cnt;
    __syncwarp();
    const int n_valid = hist[kBins];
#pragma unroll
    for (int k = 0; k < kCarRounds; k++)
      if (k * 32 < items) {
        const int pos = hist[key[k] & 0xff] + (key[k] >> 8);
        if (pos < 256) order[pos] = (unsigned char)(k * 32 + lane);
      }
    __syncwarp();
    // ---- match them, 32 of similar walk length at a time; results replace the inputs
    for (int gi = lane; gi < n_valid; gi += 32) {
      const int i = order[gi];
      const int fl = (int)(((unsigned)i * g.magic) >> 16);
      RefState rs;
      rs.wp = fwp[fl];
      rs.ratio[0] = fr0[fl];
      rs.ratio[1] = fr1[fl];
      rs.ratio[2] = fr2[fl];
      const CarRes r = car_slot(m, rs, in, cb0 + i, car0[i], car1[i], car2[i], car3[i]);
      store_car(out, cb0 + i, r);
      // its share of the frame's reductions, evaluated here where every lane has a car
      const double dt0 = fnp[fl] ? PP_PREV_KEEP / 50.0 : 0.0;
      const double s0 = r.s + r.vs * dt0;  // Car::predicted_s (:67)
      const double d0 = r.d + r.vd * dt0;  // Car::predicted_d (:70)
      double lane_speed = 0;
      unsigned fw = 0;
      if (r.lane >= 0) {
        const double es = fes[fl];
        const CarFacts cf = lane_car_facts(cfg, racc, r.lane, s0, r.vs, fel[fl], ftl[fl], es, fevs[fl]);
        lane_speed = cf.lane_speed;
        fw = cf.flags | (cf.closes ? kFactCloses : 0u);
        if (s0 > es && fabs(d0 - fed[fl]) < 3) fw |= kFactOwn;             // :1392
        if (s0 >= es - cfg.car_length - cfg.safety_distance) {             // :1402
#pragma unroll
          for (int l = 0; l < 3; l++)
            if (fabs(d0 - lane_center_offset(l)) < 3) fw |= kFactTl0 << l;
        }
      }
      car0[i] = s0;
      car2[i] = lane_speed;
      *reinterpret_cast<int2 *>(car3 + i) = make_int2(r.lane, (int)fw);
    }
    __syncwarp();
    // ---- per-frame reductions (:377-445, :1388-1410).  Lanes fl G .. fl G + G - 1 share the
    // cars of frame fl (lane k takes j = k mod G), visiting them from a lane-dependent start
    // (spreads the banks); every reduction is order-free, so the partial results merge with a
    // butterfly and lane k = 0 stores the frame's outcome.
    {
      const int Cg = g.Cg;
      const int fl = lane / G, k = lane - fl * G;
      const bool act = fl < nf;
      const int64_t f = f0 + (act ? fl : 0);
      uint32_t pflags = 0;
      Behav bp;
      behav_init(bp, cfg);
      if (act) {
        const double e_s = fes[fl];
        const int e_nc = fnc[fl];
        int j = (fl * G) % Cg + k;
        if (j >= Cg) j -= Cg;
        const int base = fl * mc;
        const int32_t *ids = in.car_id + cb0 + base;
        for (int q = 0; q < Cg; q += G) {
          if (j < e_nc) {
            const int2 w = *reinterpret_cast<const int2 *>(car3 + base + j);
            const unsigned fw = (unsigned)w.y;
            if (w.x < 0) {  // :1336-1340 dropped from the map
              pflags |= PP_F_CAR_DROPPED;
            } else {
              const double s0 = car0[base + j];
              const int id = ids[j];
              pflags |= fw & kFactFlags;
              lane_stats_take(bp.ls, id, w.x, s0, s0 > e_s, car2[base + j], (fw & kFactCloses) != 0);
              if (fw & kFactOwn) cand_offer(bp.own, s0, id, j);
              if (fw & kFactTl0) cand_offer(bp.tl0, s0, id, j);
              if (fw & (kFactTl0 << 1)) cand_offer(bp.tl1, s0, id, j);
              if (fw & (kFactTl0 << 2)) cand_offer(bp.tl2, s0, id, j);
            }
          }
          j += G;
          if (j >= Cg) j -= Cg;
        }
      }
      for (int o = 1; o < G; o <<= 1) behav_merge_xor(bp, pflags, o);
      if (act && k == 0) behav_store(sc, f, bp, pflags);
    }
    fence_async_smem();  // results were written where the next tile's bulk copies land
    __syncwarp();
  }
}

// Decision, trajectory set-up and spline fit, one thread per frame, tiles of kBlock frames:
// the tile's previous points arrive by one bulk copy per coordinate while the threads reduce
// their cars and decide, and the kept points of the result (= those previous points, :578)
// leave from the same tile by bulk copies — as strided loads and stores of every lane's own
// 80-byte rows these were 10 % of this kernel's stall samples and 0.1 ms per 1M frames.
// kBehav: the reductions were done by k_cars_t (variant 3), else they run here over the
// car-major scratch of k_cars.  Frames whose trajectory is the ordinary spline emission hand
// their state to k_emit; the rest (angle-based generator, :848) are queued for k_fallback.
template <bool kBehav>
__global__ void __launch_bounds__(kBlock, PP_DECIDE_MINB)
k_decide_t(const double *__restrict__ map_table, int n_wp, const __grid_constant__ pp_config cfg,
           const __grid_constant__ pp_frames in, const __grid_constant__ pp_plans out,
           const __grid_constant__ Scratch sc, int64_t n, int bulk_in, int bulk_out,
           const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_y) {
  // bulk_out: 0 = the kept points go out by ordinary stores, 1 = one 80-byte bulk copy per lane
  // and coordinate, 2 = ONE 2-D tensor-map store per tile and coordinate (tm_x / tm_y describe
  // next_x / next_y of this chunk as [n][50] with a box of [128 rows][10 columns]; a tensor
  // copy wants its shared-memory side on a 128-byte boundary: s_px / s_py are at 35,840 and
  // 46,080 bytes of a 128-byte aligned array)
  extern __shared__ __align__(128) double s_dyn[];
  double *s_rows = s_dyn;                                      // [PPD_SWEEP_ROWS * PPD_TAILK][kBlock]
  double *s_px = s_dyn + PPD_SWEEP_ROWS * PPD_TAILK * kBlock;  // [kBlock][10]
  double *s_py = s_px + kBlock * PP_PREV_KEEP;
  __shared__ __align__(8) unsigned long long s_bar;
  const unsigned bar = smem_addr(&s_bar);
  if (threadIdx.x == 0) mbar_init(bar, 1);
  __syncthreads();
  MapView m;
  m.t = map_table + PPD_PAD * PP_MAP_STRIDE;
  m.n = n_wp;
  m.pad_lo = n_wp < PPD_PAD ? n_wp : PPD_PAD;
  const int64_t n_tiles = (n + kBlock - 1) / kBlock;
  long long xacc = 0;  // checksum of the kept points (= the stored previous points, :578)
  unsigned phase = 0;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t f0 = tile * kBlock;
    const int nf = (int)((n - f0) < kBlock ? (n - f0) : kBlock);
    const unsigned bytes = (unsigned)nf * PP_PREV_KEEP * 8u;  // a multiple of 16
    if (bulk_in && threadIdx.x == 0) {
      mbar_expect_tx(bar, 2u * bytes);
      bulk_g2s(smem_addr(s_px), in.prev_x + f0 * PP_PREV_KEEP, bytes, bar);
      bulk_g2s(smem_addr(s_py), in.prev_y + f0 * PP_PREV_KEEP, bytes, bar);
    }
    // (the decision needs nothing of the tile: it runs while the copy is in flight)
    const int64_t f = f0 + threadIdx.x;
    const bool own = threadIdx.x < nf;
    FrameCtx c;
    Decision d;
    if (own) {
      load_ctx(sc, f, c);
      uint32_t flags = c.flags;
      const int tl_in = in.target_lane_in[f];
      Behav b;
      if (kBehav)
        behav_load(sc, cfg, f, b, flags);
      else
        reduce_cars(cfg, in, sc, f, c, tl_in, b, flags);
      d = stage_decide(cfg, in, out, f, c, b, tl_in, flags);
    }
    if (bulk_in) {
      mbar_wait(bar, phase);
      phase ^= 1;
    } else {
      for (int i = threadIdx.x; i < nf * PP_PREV_KEEP; i += kBlock) {
        s_px[i] = in.prev_x[f0 * PP_PREV_KEEP + i];
        s_py[i] = in.prev_y[f0 * PP_PREV_KEEP + i];
      }
      __syncthreads();
    }
    if (bulk_out == 2 && threadIdx.x == 0) {
      // result_points = prev_trajectory (:578) for the whole tile at once: columns [0, 10) of
      // rows f0 .. f0 + 127 (rows past the chunk are clipped by the tensor map).  A frame
      // WITHOUT a previous path gets its stale input row here; every one of its 50 columns is
      // written afterwards by the kernel that emits its points (k_emit / k_fallback / k_slow).
      fence_async_smem();
      tensor_s2g_2d(&tm_x, 0, (int)f0, smem_addr(s_px));
      tensor_s2g_2d(&tm_y, 0, (int)f0, smem_addr(s_py));
      bulk_commit();
    }
    if (own) {
      const double *px = s_px + threadIdx.x * PP_PREV_KEEP;
      const double *py = s_py + threadIdx.x * PP_PREV_KEEP;
      uint32_t flags = d.flags;
      double *gx = out.next_x + f * PP_PATH_LEN, *gy = out.next_y + f * PP_PATH_LEN;
      if (c.nprev) {  // result_points = prev_trajectory (:578): straight from the staged tile
        if (bulk_out == 1) {
          bulk_s2g(gx, smem_addr(px), PP_PREV_KEEP * 8);
          bulk_s2g(gy, smem_addr(py), PP_PREV_KEEP * 8);
          bulk_commit();
        }
        if (sc.xsum) {
#pragma unroll
          for (int h = 0; h < PP_PREV_KEEP / 2; h++) {
            const double2 qx = reinterpret_cast<const double2 *>(px)[h];
            const double2 qy = reinterpret_cast<const double2 *>(py)[h];
            xacc += fx_point(qx.x, qy.x) + fx_point(qx.y, qy.y);
          }
        }
      }
      double *e = sc.est + f;
      KnotSweep sw;
      sw.init(s_rows + threadIdx.x, kBlock, e, sc.n, kEstHead);
      TrajFrame tf;
      traj_setup<true>(m, cfg, c.rs, px, py, c.nprev, c.x, c.y, in.ego_yaw_deg[f], d.target_lane,
                       c.d, c.vd, d.sc, bulk_out ? nullptr : gx, bulk_out ? nullptr : gy, flags, sw,
                       tf);
      e[0 * sc.n] = d.sc.start;
      e[1 * sc.n] = d.sc.target;
      e[2 * sc.n] = d.sc.time;
      e[3 * sc.n] = tf.cx;
      e[4 * sc.n] = tf.cy;
      e[5 * sc.n] = tf.ca;
      e[6 * sc.n] = tf.sa;
      sc.e_np[f] = tf.np;
      if (tf.fallback) {  // :848 the angle-based generator: its own (converged) kernel
#pragma unroll
        for (int k = 0; k < 6; k++) {
          e[(kEstHead + k) * sc.n] = tf.cpx[k];
          e[(kEstHead + 6 + k) * sc.n] = tf.cpy[k];
        }
        sc.e_nk[f] = kEstFallback | tf.ncp;
        sc.e_flags[f] = flags | PP_F_FALLBACK;
        sc.slow_qa[atomicAdd(sc.slow_na, 1)] = (int32_t)f;
      } else {
        const int r0 = sw.r0;
        const int cnt = sw.solve(tf.nk);  // a, b, c of the reachable rows -> emission state
        sc.e_nk[f] = cnt | (r0 > 0 ? kEstPartial : 0);
        sc.e_flags[f] = flags;
      }
      if (bulk_out == 1) bulk_wait_read();  // the tile is overwritten by the next load
    }
    if (bulk_out == 2 && threadIdx.x == 0) bulk_wait_read();
    fence_async_smem();
    __syncthreads();
  }
  if (bulk_out) bulk_wait_all();
  if (sc.xsum) xsum_commit(sc.xsum, xacc);
}

// The complete path for the frames k_emit gave up on (tiled pipeline): re-planned from their inputs alone
// (a few hundred per million; every output is rewritten with the same values, the trajectory
// by the complete emission loop), one frame per warp.
__global__ void __launch_bounds__(kBlock)
k_slow_t(const double *__restrict__ map_table, int n_wp, const __grid_constant__ pp_config cfg,
         const __grid_constant__ pp_frames in, const __grid_constant__ pp_plans out,
         unsigned long long *xsum, const int32_t *__restrict__ queue,
         const int32_t *__restrict__ queue_n) {
  const int count = *queue_n;
  const int per_block = kBlock / kSlowSpread;
  if ((int64_t)blockIdx.x * per_block >= count) return;
  extern __shared__ __align__(16) double s_map[];
  const MapView m = stage_map(s_map, map_table, n_wp);
  if (threadIdx.x % kSlowSpread) return;
  const int64_t stride = (int64_t)gridDim.x * per_block;
  for (int64_t q = (int64_t)blockIdx.x * per_block + threadIdx.x / kSlowSpread; q < count;
       q += stride) {
    const int64_t f = queue[q];
    plan_one_frame(m, cfg, in, out, f);
    if (xsum) {  // the new points (the kept ones were counted by k_decide_t)
      long long xacc = 0;
      const int np = out.n_points[f];
      const int nprev = in.prev_n[f] >= PP_PREV_KEEP ? PP_PREV_KEEP : 0;
      for (int i = nprev; i < np; i++)
        xacc += fx_point(out.next_x[f * PP_PATH_LEN + i], out.next_y[f * PP_PATH_LEN + i]);
      if (xacc) atomicAdd(xsum, (unsigned long long)xacc);
    }
  }
}

// ---- aggregate statistics (SURVEY §8e): exact int64 sums -----------------
// HBM bound (re-reads the plans: 828 B/frame).  The trajectories are read as one
// flat array (coalesced; the owning frame's n_points masks the padding), the
// per-frame scalars in a second pass with warp ballots instead of one atomic per
// frame and flag.
__device__ __forceinline__ unsigned long long warp_sum(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}
__global__ void __launch_bounds__(256)
stats_kernel(const __grid_constant__ pp_plans p, int64_t n, unsigned long long *stats,
             bool with_points) {
  __shared__ unsigned long long s_acc[PP_STATS_LEN];
  for (int i = threadIdx.x; i < PP_STATS_LEN; i += blockDim.x) s_acc[i] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  // pass 1: fixed-point (1/256 m) checksum of every emitted point: order-independent.
  // Four independent elements per trip and unconditional loads (the padding is valid memory,
  // n_points only masks it afterwards) keep enough requests in flight to reach HBM speed.
  long long xs = 0;
  const bool wide = (((uintptr_t)p.next_x | (uintptr_t)p.next_y) & 15) == 0;
  constexpr int kU = 4;
  auto add_point = [&](double x, double y, bool live) {
    if (live) xs += fx_point(x, y);
  };
  if (!with_points) {
    // the pipeline accumulated the checksum while it produced the points
  } else if (wide) {  // two points per load: a row holds an even number of points
    const int64_t total = n * (PP_PATH_LEN / 2);
    const double2 *px = reinterpret_cast<const double2 *>(p.next_x);
    const double2 *py = reinterpret_cast<const double2 *>(p.next_y);
    for (int64_t e0 = tid; e0 < total; e0 += stride * kU) {
      double2 xv[kU], yv[kU];
      int lim[kU], idx[kU];
#pragma unroll
      for (int u = 0; u < kU; u++) {
        const int64_t e = e0 + u * stride;
        const bool in = e < total;
        const int64_t ec = in ? e : 0;
        const int64_t f = ec / (PP_PATH_LEN / 2);
        idx[u] = 2 * (int)(ec - f * (PP_PATH_LEN / 2));
        xv[u] = px[ec];
        yv[u] = py[ec];
        lim[u] = in ? p.n_points[f] : 0;
      }
#pragma unroll
      for (int u = 0; u < kU; u++) {
        add_point(xv[u].x, yv[u].x, idx[u] < lim[u]);
        add_point(xv[u].y, yv[u].y, idx[u] + 1 < lim[u]);
      }
    }
  } else {
    const int64_t total = n * PP_PATH_LEN;
    for (int64_t e0 = tid; e0 < total; e0 += stride * kU) {
      double xv[kU], yv[kU];
      int lim[kU], idx[kU];
#pragma unroll
      for (int u = 0; u < kU; u++) {
        const int64_t e = e0 + u * stride;
        const bool in = e < total;
        const int64_t ec = in ? e : 0;
        const int64_t f = ec / PP_PATH_LEN;
        idx[u] = (int)(ec - f * PP_PATH_LEN);
        xv[u] = p.next_x[ec];
        yv[u] = p.next_y[ec];
        lim[u] = in ? p.n_points[f] : 0;
      }
#pragma unroll
      for (int u = 0; u < kU; u++) add_point(xv[u], yv[u], idx[u] < lim[u]);
    }
  }
  const unsigned long long xw = warp_sum((unsigned long long)xs);
  if (lane == 0 && xw) atomicAdd(&s_acc[PP_STAT_XSUM], xw);
  // pass 2: per-frame counters.  Whole warps iterate together (ballots need every lane).
  const int64_t n_round = (n + 31) / 32 * 32;
  for (int64_t f = tid; f < n_round; f += stride) {
    const bool live = f < n;
    const int np = live ? p.n_points[f] : 0;
    const int tl = live ? p.target_lane[f] : -1, el = live ? p.ego_lane[f] : -1;
    const uint32_t fl = live ? p.flags[f] : 0u;
    const unsigned long long pts = warp_sum((unsigned long long)np);
    const unsigned m_live = __ballot_sync(0xffffffffu, live);
    const unsigned m_chg = __ballot_sync(0xffffffffu, live && tl != el);
    unsigned m_tl[3], m_el[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
      m_tl[k] = __ballot_sync(0xffffffffu, tl == k);
      m_el[k] = __ballot_sync(0xffffffffu, el == k);
    }
    // lane b counts flag bit b
    unsigned my_flag = 0;
#pragma unroll
    for (int b = 0; b < PP_NUM_FLAGS; b++) {
      const unsigned mb = __ballot_sync(0xffffffffu, (fl >> b) & 1u);
      if (lane == b) my_flag = mb;
    }
    if (lane < PP_NUM_FLAGS && my_flag)
      atomicAdd(&s_acc[PP_STAT_FLAG0 + lane], (unsigned long long)__popc(my_flag));
    if (lane == 0) {
      atomicAdd(&s_acc[PP_STAT_FRAMES], (unsigned long long)__popc(m_live));
      atomicAdd(&s_acc[PP_STAT_POINTS], pts);
      atomicAdd(&s_acc[PP_STAT_LANE_CHANGES], (unsigned long long)__popc(m_chg));
#pragma unroll
      for (int k = 0; k < 3; k++) {
        atomicAdd(&s_acc[PP_STAT_TARGET_LANE0 + k], (unsigned long long)__popc(m_tl[k]));
        atomicAdd(&s_acc[PP_STAT_EGO_LANE0 + k], (unsigned long long)__popc(m_el[k]));
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < PP_STATS_LEN; i += blockDim.x)
    if (s_acc[i]) atomicAdd(&stats[i], s_acc[i]);
}

// process-wide knobs (tests, bench.py, profiles/): plain loads and stores of an atomic
std::atomic<int> g_variant{0};
std::atomic<int> g_sm_count{0};

// ---- side stream for the rare-frame kernel (one per host thread and device)
struct Side {
  int dev = -1;
  cudaStream_t st = nullptr;
  cudaEvent_t ev_a = nullptr, ev_b = nullptr, ev_join = nullptr;
  cudaEvent_t ev_done = nullptr;  // the side work of this stream's last chunk has finished
  int ensure() {
    int d = 0;
    if (cudaGetDevice(&d) != cudaSuccess) return PP_E_CUDA;
    if (st && d == dev) return PP_OK;
    release();
    if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&ev_a, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ev_b, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ev_done, cudaEventDisableTiming) != cudaSuccess) {
      cudaError_t e = cudaGetLastError();
      ppi::set_cuda_error("side stream", (int)e, cudaGetErrorString(e));
      release();
      return PP_E_CUDA;
    }
    dev = d;
    return PP_OK;
  }
  void release() {
    if (ev_a) cudaEventDestroy(ev_a);
    if (ev_b) cudaEventDestroy(ev_b);
    if (ev_join) cudaEventDestroy(ev_join);
    if (ev_done) cudaEventDestroy(ev_done);
    ev_done = nullptr;
    if (st) cudaStreamDestroy(st);
    ev_a = ev_b = ev_join = nullptr;
    st = nullptr;
    dev = -1;
  }
  // not destroyed at thread exit: the CUDA context may already be gone by then
};
// One side stream per caller stream (per host thread): callers that drive several streams at
// once — the rollout engine's groups — must not serialise on each other's rare-frame kernels.
constexpr int kMaxSides = 16;
struct SideSlot {
  cudaStream_t owner = nullptr;
  bool used = false;
  Side side;
};
thread_local SideSlot t_sides[kMaxSides];

Side &side_for(cudaStream_t st) {
  for (int i = 0; i < kMaxSides; i++)
    if (t_sides[i].used && t_sides[i].owner == st) return t_sides[i].side;
  for (int i = 0; i < kMaxSides; i++)
    if (!t_sides[i].used) {
      t_sides[i].used = true;
      t_sides[i].owner = st;
      return t_sides[i].side;
    }
  return t_sides[0].side;  // more caller streams than slots: share (still correct, ordered by events)
}

// ---- pipes: a batch of several chunks is planned on kMaxPipes internal streams at once
// (chunk i on pipe i % pipes).  Each kernel of the pipeline is sized for the whole GPU, but its
// last wave and its divergent tails leave SMs idle; with a second chunk in flight those slots
// run the other chunks' kernels (measured per 1M frames, DESIGN.md §3: 3.13 ms with one pipe,
// 2.64 with two, 2.51 with four chunks of 262,144 frames in flight; more or smaller chunks do
// not help).
constexpr int kMaxPipes = 8;
struct Pipes {
  int dev = -1;
  cudaStream_t st[kMaxPipes] = {};
  cudaEvent_t done[kMaxPipes] = {};
  cudaEvent_t fork = nullptr;
  int ensure() {
    int d = 0;
    if (cudaGetDevice(&d) != cudaSuccess) return PP_E_CUDA;
    if (fork && d == dev) return PP_OK;
    release();  // (streams and events of another device: the thread moved on)
    for (int i = 0; i < kMaxPipes; i++)
      if (cudaStreamCreateWithFlags(&st[i], cudaStreamNonBlocking) != cudaSuccess ||
          cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming) != cudaSuccess)
        return PP_E_CUDA;
    if (cudaEventCreateWithFlags(&fork, cudaEventDisableTiming) != cudaSuccess) return PP_E_CUDA;
    dev = d;
    return PP_OK;
  }
  void release() {
    for (int i = 0; i < kMaxPipes; i++) {
      if (done[i]) cudaEventDestroy(done[i]);
      if (st[i]) cudaStreamDestroy(st[i]);
      done[i] = nullptr;
      st[i] = nullptr;
    }
    if (fork) cudaEventDestroy(fork);
    fork = nullptr;
    dev = -1;
    cudaGetLastError();
  }
};
thread_local Pipes t_pipes;

int env_int(const char *name, int dflt, int lo, int hi) {
  const char *v = getenv(name);
  if (!v || !*v) return dflt;
  const int k = atoi(v);
  return k < lo ? lo : (k > hi ? hi : k);
}

// ---- optional per-phase timing (bench.py / profiles): CUDA events recorded on
// the caller's stream around every kernel of the pipeline.
constexpr int kPhases = 5;  // prep, cars, decide, emit, slow
constexpr int kMaxTimedChunks = 4096;
std::atomic<bool> g_phase_timing{false};
struct PhaseEvents {
  cudaEvent_t ev[kPhases + 1];
};
std::mutex g_phase_mu;                    // guards the two vectors (callers plan from any thread)
std::vector<PhaseEvents> g_phase_events;  // one entry per chunk launched since the last read
std::vector<PhaseEvents> g_phase_pool;    // recycled events

void phase_mark(const PhaseEvents *pe, int i, cudaStream_t st) {
  if (pe) cudaEventRecord(pe->ev[i], st);
}
// (returns a copy: the vector may grow under another thread's chunk)
bool phase_begin(PhaseEvents &pe) {
  if (!g_phase_timing.load(std::memory_order_relaxed)) return false;
  std::lock_guard<std::mutex> lk(g_phase_mu);
  if ((int)g_phase_events.size() >= kMaxTimedChunks) return false;
  if (!g_phase_pool.empty()) {
    pe = g_phase_pool.back();
    g_phase_pool.pop_back();
  } else {
    for (int i = 0; i <= kPhases; i++)
      if (cudaEventCreate(&pe.ev[i]) != cudaSuccess) return false;
  }
  g_phase_events.push_back(pe);
  return true;
}

int sm_count() {
  int n = g_sm_count.load(std::memory_order_relaxed);
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
    g_sm_count.store(n, std::memory_order_relaxed);
  }
  return n;
}

int check_launch(const char *what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    ppi::set_cuda_error(what, (int)e, cudaGetErrorString(e));
    return PP_E_CUDA;
  }
  return PP_OK;
}

int stats_grid(int64_t n_frames) {
  const int64_t want = (n_frames * PP_PATH_LEN + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 8;
  return (int)(want < cap ? want : cap);
}

// persistent grid: enough blocks for `items`, capped at a whole number of waves
int grid_for(int64_t items, int blocks_per_sm) {
  const int64_t want = (items + kBlock - 1) / kBlock;
  const int64_t cap = (int64_t)sm_count() * blocks_per_sm;
  return (int)(want < cap ? want : cap);
}

// Tile geometry of k_cars_t for `mc` car slots per frame (see CarsGeom).
CarsGeom cars_geom(int mc, const pp_frames &in, int max_items) {
  CarsGeom g;
  const int c1 = mc > 0 ? mc : 1;
  int F = max_items / c1;
  F = F < 1 ? 1 : (F > 32 ? 32 : F);
  if (((F * mc) & 1) && F > 1) F--;  // an even number of car slots per tile: 16-byte granules
  g.F = F;
  int G = 1;
  while (G * 2 * F <= 32 && G * 2 <= c1) G *= 2;
  g.G = G;
  g.T = (F * mc + 1) & ~1;
  if (g.T < 2) g.T = 2;
  g.Cg = (c1 + G - 1) / G * G;
  g.warp_bytes = cars_warp_bytes(g.T, g.F);
  g.magic = (65536u + (unsigned)c1 - 1u) / (unsigned)c1;
  g.bulk = mc > 0 && aligned16(in.car_x) && aligned16(in.car_y) && aligned16(in.car_vx) &&
           aligned16(in.car_vy) && ((F * mc) % 2 == 0);
  return g;
}

template <int kThreads>
int launch_cars(const pp_map *map, const pp_config &cfg, const pp_frames &fin, const pp_plans &fout,
                const Scratch &sc, int64_t cnt, const CarsGeom &g, size_t smem_map,
                cudaStream_t st) {
  const size_t smem = smem_map + (size_t)(kThreads / 32) * g.warp_bytes;
  // (the opt-in limit is per function and device; raised whenever a call needs more)
  static std::atomic<size_t> granted[64];
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || granted[dev].load(std::memory_order_relaxed) < smem) {
    if (cudaFuncSetAttribute(k_cars_t<kThreads>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)smem) != cudaSuccess)
      return check_launch("cudaFuncSetAttribute(k_cars_t)");
    if (dev >= 0 && dev < 64) granted[dev].store(smem, std::memory_order_relaxed);
  }
  const int64_t n_tiles = (cnt + g.F - 1) / g.F;
  const int64_t want = (n_tiles + kThreads / 32 - 1) / (kThreads / 32);
  const int grid = (int)(want < sm_count() ? want : sm_count());
  k_cars_t<kThreads><<<grid, kThreads, smem, st>>>(map->dev_table, map->n, cfg, fin, fout, sc, cnt, g);
  return PP_OK;
}

using ppi::offset_frames;
using ppi::offset_plans;

constexpr int64_t kPipeChunk = 1 << 18;  // frames per scratch buffer (≈ 155 MB at 12 cars)
constexpr int64_t kFusedBelow = 1536;    // auto: batches this small take the warp-per-frame kernel
                                         // (profiles/r2_latency.log: 82 us at 1,024 frames against
                                         // 124 us for the pipeline; 246 against 131 at 4,095)

// 2-D tensor map of a plan array [rows][50] of doubles with a box of [kBlock rows][10 columns]
// (the kept points of a k_decide_t tile).  The encoder lives in the driver library; it is
// fetched through the runtime, so nothing links against libcuda.
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *,
                                  const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                  const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn tensor_encoder() {
  static const EncodeTiledFn fn = [] {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    cudaGetLastError();
    return (EncodeTiledFn)p;
  }();
  return fn;
}
bool kept_points_map(CUtensorMap &tm, double *base, int64_t rows) {
  // (a closed-loop run asks for the same few (array, rows) pairs every tick: keep the last ones)
  struct Entry {
    double *base = nullptr;
    int64_t rows = 0;
    CUtensorMap tm;
  };
  constexpr int kKeep = 32;
  thread_local Entry cache[kKeep];
  thread_local int next = 0;
  for (int i = 0; i < kKeep; i++)
    if (cache[i].base == base && cache[i].rows == rows) {
      tm = cache[i].tm;
      return true;
    }
  const EncodeTiledFn enc = tensor_encoder();
  if (!enc || rows <= 0) return false;
  const cuuint64_t gdim[2] = {PP_PATH_LEN, (cuuint64_t)rows};
  const cuuint64_t gstride[1] = {PP_PATH_LEN * sizeof(double)};
  const cuuint32_t box[2] = {PP_PREV_KEEP, kBlock};
  const cuuint32_t estr[2] = {1, 1};
  if (enc(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, base, gdim, gstride, box, estr,
          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
    return false;
  cache[next].base = base;
  cache[next].rows = rows;
  cache[next].tm = tm;
  next = (next + 1) % kKeep;
  return true;
}

template <class K>
int ensure_smem(K kernel, size_t smem) {
  // (the 48 KB default limit counts static shared memory too: k_cars has 2.5 KB of it)
  if (smem > 40 * 1024) {
    if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) !=
        cudaSuccess)
      return check_launch("cudaFuncSetAttribute");
  }
  return PP_OK;
}

}  // namespace

extern "C" int pp_set_kernel_variant(int variant) {
  if (variant < 0 || variant > 4) return PP_E_ARG;
  g_variant = variant;
  return PP_OK;
}

// frames per chunk and chunks in flight (PP_PIPE_CHUNK / PP_PIPES: tuning experiments)
static int pipe_count();
// frames per chunk for a batch of n: at most PP_PIPE_CHUNK (262,144), and small enough that a
// mid-sized batch still splits into one chunk per pipe (but not below 32,768 frames)
static int64_t chunk_for(int64_t n, int pipes) {
  static const int64_t cap = env_int("PP_PIPE_CHUNK", (int)kPipeChunk, 4096, 1 << 22);
  const int64_t floor_ = 32768 < cap ? 32768 : cap;
  int64_t c = (n + pipes - 1) / pipes;
  c = (c + 1023) / 1024 * 1024;
  if (c < floor_) c = floor_;
  if (c > cap) c = cap;
  return c < n ? c : n;
}
static std::atomic<int> g_pipes_override{0};  // pp_set_pipes
static int pipe_count() {
  static const int v = env_int("PP_PIPES", 4, 1, kMaxPipes);
  const int o = g_pipes_override.load(std::memory_order_relaxed);
  return o > 0 ? o : v;
}

// Bytes of scratch the pipeline needs for a batch (0 for batches the fused kernel takes).
// (a caller that brings its own scratch drives its own concurrency: one chunk in flight)
size_t ppi::plan_scratch_bytes(int64_t n_frames, int max_cars) {
  const int variant = g_variant.load(std::memory_order_relaxed);
  if (n_frames <= 0 || variant == 1 || variant == 4 || (variant == 0 && n_frames < kFusedBelow))
    return 0;
  const int64_t chunk = chunk_for(n_frames, 1);
  const int64_t n_chunks = (n_frames + chunk - 1) / chunk;
  const int n_buf = 1;
  size_t scratch = 0;
  carve_chunk(nullptr, variant == 3, chunk, max_cars, &scratch);
  return n_buf * scratch + (size_t)n_frames * 2 * sizeof(int32_t) +
         (size_t)n_chunks * 2 * sizeof(int32_t) + 256;
}

extern "C" int pp_plan_batch(const pp_map *map, const pp_config *cfg, const pp_frames *in,
                             const pp_plans *out, int64_t n_frames, void *cuda_stream) {
  return ppi::plan_batch_scratch(map, cfg, in, out, n_frames, cuda_stream, nullptr, nullptr);
}

// pp_plan_batch followed by pp_stats_batch as one call: the statistics of a chunk are taken on
// the chunk's own internal stream as soon as it is planned, so the HBM-bound statistics pass
// shares the GPU with the FP64-bound kernels of the other chunks instead of running alone.
extern "C" int pp_plan_stats_batch(const pp_map *map, const pp_config *cfg, const pp_frames *in,
                                   const pp_plans *out, int64_t n_frames, int64_t *stats_dev,
                                   void *cuda_stream) {
  if (!stats_dev) return PP_E_ARG;
  return ppi::plan_batch_scratch(map, cfg, in, out, n_frames, cuda_stream, nullptr, stats_dev);
}

// pp_plan_batch with the scratch supplied by the caller (plan_scratch_bytes; nullptr: taken
// from the stream-ordered pool).  The rollout engine owns its scratch so that a tick is pure
// kernel / memset / event work and can be replayed as a CUDA graph.
bool ppi::plan_adds_checksum(int64_t n_frames) {
  const int variant = g_variant.load(std::memory_order_relaxed);
  return !(variant == 1 || variant == 4 || (variant == 0 && n_frames < kFusedBelow));
}

int ppi::plan_batch_scratch(const pp_map *map, const pp_config *cfg, const pp_frames *in,
                            const pp_plans *out, int64_t n_frames, void *cuda_stream,
                            char *caller_scratch, int64_t *stats_dev,
                            unsigned long long *xsum_add) {
  if (!map || !cfg || !in || !out || n_frames < 0) return PP_E_ARG;
  int rc0;
  if (stats_dev &&
      cudaMemsetAsync(stats_dev, 0, PP_STATS_LEN * sizeof(int64_t), (cudaStream_t)cuda_stream) !=
          cudaSuccess)
    return check_launch("pp_plan_stats_batch memset");
  if ((rc0 = ppi::check_map_device(map, "pp_plan_batch")) != PP_OK) return rc0;
  if (in->max_cars < 0 || in->max_cars > PP_MAX_CARS) return PP_E_RANGE;
  if (!in->ego_x || !in->ego_y || !in->ego_yaw_deg || !in->ego_speed_mph || !in->prev_n ||
      !in->prev_x || !in->prev_y || !in->target_lane_in || !in->n_cars)
    return PP_E_ARG;
  if (in->max_cars > 0 && (!in->car_id || !in->car_x || !in->car_y || !in->car_vx || !in->car_vy))
    return PP_E_ARG;
  if (!out->next_x || !out->next_y || !out->n_points || !out->ego_lane || !out->ref_wp ||
      !out->target_lane || !out->flags)
    return PP_E_ARG;
  if (n_frames == 0) return PP_OK;
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const size_t smem = map_stage_bytes(map->n);
  if (smem > 200 * 1024) return PP_E_RANGE;
  int rc;
  if ((rc = ensure_smem(plan_fused, smem)) != PP_OK) return rc;
  if ((rc = ensure_smem(plan_warp, smem)) != PP_OK) return rc;
  if ((rc = ensure_smem(k_prep, smem)) != PP_OK) return rc;
  if ((rc = ensure_smem(k_cars<kTileKBig>, smem)) != PP_OK) return rc;
  if ((rc = ensure_smem(k_cars<kTileKSmall>, smem)) != PP_OK) return rc;
  if ((rc = ensure_smem(k_slow, smem)) != PP_OK) return rc;
  const size_t smem_emit = (size_t)5 * PPD_TAILK * kBlock * sizeof(double);
  if ((rc = ensure_smem(k_emit<ArrayOut, false>, smem_emit)) != PP_OK) return rc;
  if ((rc = ensure_smem(k_emit<PairOut, false>, smem_emit)) != PP_OK) return rc;
  if ((rc = ensure_smem(k_emit<ArrayOut, true>, smem_emit)) != PP_OK) return rc;
  if ((rc = ensure_smem(k_emit<PairOut, true>, smem_emit)) != PP_OK) return rc;
  const bool paired = (((uintptr_t)out->next_x | (uintptr_t)out->next_y) & 15) == 0;
  const int variant = g_variant.load(std::memory_order_relaxed);  // one reading per call
  const bool tiled = variant == 3;  // k_cars_t + reduced Behav in the scratch
  const size_t smem_tile =
      (size_t)(5 * PPD_TAILK * kBlock + 2 * kBlock * PP_PREV_KEEP) * sizeof(double);
  static_assert(PPD_SWEEP_ROWS == 5, "k_decide_t tile size");
  if ((rc = ensure_smem(k_decide_t<false>, smem_tile)) != PP_OK) return rc;
  if ((rc = ensure_smem(k_decide_t<true>, smem_tile)) != PP_OK) return rc;
  if ((rc = ensure_smem(k_slow_t, smem)) != PP_OK) return rc;
  // kept points out of k_decide_t: 2 = one tensor-map store per tile, 1 = a bulk copy per lane,
  // 0 = ordinary stores (experiments; unaligned rows always take 0)
  static const int decide_bulk_out = env_int("PP_DECIDE_BULK_OUT", 2, 0, 2);
  // persistent grids: blocks per SM each kernel may occupy (a smaller share leaves room for the
  // kernels of the other chunks in flight; profiles/r2_grids.log)
  static const int decide_blocks = env_int("PP_DECIDE_BLOCKS", 4, 1, 16);
  static const int prep_blocks = env_int("PP_PREP_BLOCKS", 12, 1, 16);
  static const int cars_blocks = env_int("PP_CARS_BLOCKS", 12, 1, 16);
  static const int emit_blocks = env_int("PP_EMIT_BLOCKS", 12, 1, 16);
  const int bulk_prev = aligned16(in->prev_x) && aligned16(in->prev_y);

  const bool fused = variant == 1 || variant == 4 || (variant == 0 && n_frames < kFusedBelow);
  if (fused) {
    if (variant == 1) {
      plan_fused<<<grid_for(n_frames, 8), kBlock, smem, st>>>(map->dev_table, map->n, *cfg, *in, *out,
                                                              n_frames);
    } else {  // small batches: one warp per frame
      const int64_t want = (n_frames + kBlock / 32 - 1) / (kBlock / 32);
      const int64_t cap = (int64_t)sm_count() * 4;
      plan_warp<<<(int)(want < cap ? want : cap), kBlock, smem, st>>>(map->dev_table, map->n, *cfg, *in,
                                                                     *out, n_frames);
    }
    ppi::count_launch();
    if (stats_dev) {
      stats_kernel<<<stats_grid(n_frames), 256, 0, st>>>(*out, n_frames,
                                                         (unsigned long long *)stats_dev, true);
      ppi::count_launch();
    }
    return check_launch("plan_fused");
  }

  const int mc = in->max_cars;
  const int max_pipes = caller_scratch ? 1 : pipe_count();
  const int64_t chunk = chunk_for(n_frames, max_pipes);
  {  // keep freed scratch inside the stream-ordered pool (default threshold 0 hands it back to
     // the driver at every synchronisation, which costs milliseconds per call)
    static bool pool_tuned[64] = {false};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !pool_tuned[dev]) {
      cudaMemPool_t pool;
      if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        uint64_t keep = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
      }
      cudaGetLastError();
      pool_tuned[dev] = true;
    }
  }
  // Chunks are planned on `pipes` internal streams at once (see Pipes); a single chunk runs on
  // the caller's stream.  Every pipe has its own scratch buffer and its own side stream.
  const int64_t n_chunks = (n_frames + chunk - 1) / chunk;
  const int pipes = (int)(n_chunks < max_pipes ? n_chunks : max_pipes);
  Pipes &pp_ = t_pipes;
  if (pipes > 1 && pp_.ensure() != PP_OK) return check_launch("pipe streams");
  cudaStream_t lane_st[kMaxPipes];
  Side *lane_side[kMaxPipes];
  for (int k = 0; k < pipes; k++) {
    lane_st[k] = pipes > 1 ? pp_.st[k] : st;
    lane_side[k] = &side_for(lane_st[k]);
    if ((rc = lane_side[k]->ensure()) != PP_OK) return rc;
  }
  size_t scratch = 0;
  carve_chunk(nullptr, tiled, chunk, mc, &scratch);
  const size_t queues = (size_t)n_frames * 2 * sizeof(int32_t);
  const size_t counters = (size_t)n_chunks * 2 * sizeof(int32_t);
  char *buf = caller_scratch;
  if (!buf) {
    cudaError_t e = cudaMallocAsync((void **)&buf, pipes * scratch + queues + counters + 256, st);
    if (e != cudaSuccess) {
      ppi::set_cuda_error("cudaMallocAsync(scratch)", (int)e, cudaGetErrorString(e));
      cudaGetLastError();
      return PP_E_CUDA;
    }
  }
  Scratch scs[kMaxPipes];
  for (int k = 0; k < pipes; k++)
    scs[k] = carve_chunk(buf + k * scratch, tiled, chunk, mc);
  static const int cars_items = env_int("PP_CARS_ITEMS", 256, 32, 256);
  static const int cars_threads = env_int("PP_CARS_THREADS", 0, 0, 1024);
  const CarsGeom cg = cars_geom(mc, *in, cars_items);
  // as many warps per SM as the shared memory holds (one block per SM)
  int cthreads = cars_threads;
  if (cthreads == 0) {
    const size_t room = 227 * 1024 - 1024 - smem;
    const int w = (int)(room / (size_t)cg.warp_bytes);
    cthreads = w >= 24 ? 768 : (w >= 20 ? 640 : (w >= 16 ? 512 : (w >= 12 ? 384 : 256)));
  }
  int32_t *q_base = (int32_t *)(buf + pipes * scratch);
  int32_t *n_base = (int32_t *)(buf + pipes * scratch + queues);
  cudaMemsetAsync(n_base, 0, counters + 64, st);
  if (pipes > 1) {  // fork: the pipes start after what the caller's stream has queued
    cudaEventRecord(pp_.fork, st);
    for (int k = 0; k < pipes; k++) cudaStreamWaitEvent(lane_st[k], pp_.fork, 0);
  }
  static const bool dbg = getenv("PP_DEBUG_SLOW") != nullptr;  // diagnostic: queue lengths
  rc = PP_OK;
  const int side_grid = sm_count() * 4;
  int64_t ci = 0;
  PhaseEvents pe_store;
  const PhaseEvents *pe = nullptr;
  for (int64_t lo = 0; lo < n_frames && rc == PP_OK; lo += chunk, ci++) {
    const int64_t cnt = (n_frames - lo) < chunk ? (n_frames - lo) : chunk;
    const pp_frames fin = offset_frames(*in, lo);
    const pp_plans fout = offset_plans(*out, lo, mc);
    const int k = (int)(ci % pipes);
    cudaStream_t ls = lane_st[k];
    Side &side = *lane_side[k];
    Scratch &sc = scs[k];
    sc.slow_qa = q_base + 2 * lo;  // queue entries are chunk-relative frame numbers
    sc.slow_qb = q_base + 2 * lo + cnt;
    sc.slow_na = n_base + 2 * ci;
    sc.slow_nb = n_base + 2 * ci + 1;
    sc.dbg = dbg ? n_base + 2 * n_chunks : nullptr;
    sc.xsum = stats_dev ? (unsigned long long *)stats_dev + PP_STAT_XSUM : xsum_add;
    // how the kept points leave k_decide_t (see there); the tensor maps describe THIS chunk's rows
    CUtensorMap tm_x, tm_y;
    std::memset(&tm_x, 0, sizeof tm_x);
    std::memset(&tm_y, 0, sizeof tm_y);
    int bulk_out = paired ? decide_bulk_out : 0;
    if (bulk_out == 2 &&
        !(kept_points_map(tm_x, fout.next_x, cnt) && kept_points_map(tm_y, fout.next_y, cnt)))
      bulk_out = 1;
    // the side stream may still be reading this pipe's scratch for its previous chunk
    if (ci >= pipes) cudaStreamWaitEvent(ls, side.ev_done, 0);
    pe = phase_begin(pe_store) ? &pe_store : nullptr;
    phase_mark(pe, 0, ls);
    if (tiled) {
      // (the car arrays of a chunk start on a 16-byte boundary when those of the batch do:
      // chunks are multiples of 1024 frames)
      k_prep<<<grid_for(cnt, prep_blocks), kBlock, smem, ls>>>(map->dev_table, map->n, *cfg, fin, sc, cnt);
      phase_mark(pe, 1, ls);
      if (mc > 0) {
        switch (cthreads) {
          case 768: rc = launch_cars<768>(map, *cfg, fin, fout, sc, cnt, cg, smem, ls); break;
          case 640: rc = launch_cars<640>(map, *cfg, fin, fout, sc, cnt, cg, smem, ls); break;
          case 512: rc = launch_cars<512>(map, *cfg, fin, fout, sc, cnt, cg, smem, ls); break;
          case 384: rc = launch_cars<384>(map, *cfg, fin, fout, sc, cnt, cg, smem, ls); break;
          default: rc = launch_cars<256>(map, *cfg, fin, fout, sc, cnt, cg, smem, ls); break;
        }
        if (rc != PP_OK) break;
      }
      phase_mark(pe, 2, ls);
      k_decide_t<true><<<grid_for(cnt, decide_blocks), kBlock, smem_tile, ls>>>(
          map->dev_table, map->n, *cfg, fin, fout, sc, cnt, bulk_prev, bulk_out, tm_x, tm_y);
      phase_mark(pe, 3, ls);
      cudaEventRecord(side.ev_a, ls);
      cudaStreamWaitEvent(side.st, side.ev_a, 0);
      k_fallback<<<side_grid, kBlock, 0, side.st>>>(fout, sc, sc.slow_qa, sc.slow_na);
      const int eg = grid_for(cnt, emit_blocks);
      if (paired) {
        if (sc.xsum)
          k_emit<PairOut, true><<<eg, kBlock, smem_emit, ls>>>(*cfg, fout, sc, cnt);
        else
          k_emit<PairOut, false><<<eg, kBlock, smem_emit, ls>>>(*cfg, fout, sc, cnt);
      } else {
        if (sc.xsum)
          k_emit<ArrayOut, true><<<eg, kBlock, smem_emit, ls>>>(*cfg, fout, sc, cnt);
        else
          k_emit<ArrayOut, false><<<eg, kBlock, smem_emit, ls>>>(*cfg, fout, sc, cnt);
      }
      phase_mark(pe, 4, ls);
      cudaEventRecord(side.ev_b, ls);
      cudaStreamWaitEvent(side.st, side.ev_b, 0);
      k_slow_t<<<side_grid, kBlock, smem, side.st>>>(map->dev_table, map->n, *cfg, fin, fout, sc.xsum,
                                                     sc.slow_qb, sc.slow_nb);
      cudaEventRecord(side.ev_done, side.st);
      ppi::count_launch(mc > 0 ? 6 : 5);
      if (stats_dev) {
        cudaStreamWaitEvent(ls, side.ev_done, 0);
        stats_kernel<<<stats_grid(cnt), 256, 0, ls>>>(fout, cnt, (unsigned long long *)stats_dev,
                                                      false);
        ppi::count_launch();
      }
      rc = check_launch("plan pipeline (tiled)");
      phase_mark(pe, 5, ls);
      continue;
    }
    k_prep<<<grid_for(cnt, prep_blocks), kBlock, smem, ls>>>(map->dev_table, map->n, *cfg, fin, sc, cnt);
    phase_mark(pe, 1, ls);
    if (mc > 0) {
      // (a resident warp per tile of 256: 148 SMs x 6 blocks x 4 warps)
      const bool small = cnt * mc < (int64_t)sm_count() * 6 * 4 * 32 * kTileKBig;
      if (small)
        k_cars<kTileKSmall><<<grid_for((cnt * mc + kTileKSmall - 1) / kTileKSmall, cars_blocks), kBlock,
                              smem, ls>>>(map->dev_table, map->n, fin, fout, sc, cnt);
      else
        k_cars<kTileKBig><<<grid_for((cnt * mc + kTileKBig - 1) / kTileKBig, cars_blocks), kBlock, smem,
                            ls>>>(map->dev_table, map->n, fin, fout, sc, cnt);
    }
    phase_mark(pe, 2, ls);
    k_decide_t<false><<<grid_for(cnt, decide_blocks), kBlock, smem_tile, ls>>>(
        map->dev_table, map->n, *cfg, fin, fout, sc, cnt, bulk_prev, bulk_out, tm_x, tm_y);
    phase_mark(pe, 3, ls);
    // side stream: the frames k_decide queued, concurrently with k_emit and the next chunk
    cudaEventRecord(side.ev_a, ls);
    cudaStreamWaitEvent(side.st, side.ev_a, 0);
    k_fallback<<<side_grid, kBlock, 0, side.st>>>(fout, sc, sc.slow_qa, sc.slow_na);
    const int eg = grid_for(cnt, emit_blocks);
    if (paired) {  // (a row is 400 bytes: every frame of an aligned array is aligned)
      if (sc.xsum)
        k_emit<PairOut, true><<<eg, kBlock, smem_emit, ls>>>(*cfg, fout, sc, cnt);
      else
        k_emit<PairOut, false><<<eg, kBlock, smem_emit, ls>>>(*cfg, fout, sc, cnt);
    } else {
      if (sc.xsum)
        k_emit<ArrayOut, true><<<eg, kBlock, smem_emit, ls>>>(*cfg, fout, sc, cnt);
      else
        k_emit<ArrayOut, false><<<eg, kBlock, smem_emit, ls>>>(*cfg, fout, sc, cnt);
    }
    phase_mark(pe, 4, ls);
    cudaEventRecord(side.ev_b, ls);
    cudaStreamWaitEvent(side.st, side.ev_b, 0);
    k_slow<<<side_grid, kBlock, smem, side.st>>>(map->dev_table, map->n, *cfg, fin, fout, sc,
                                                 sc.slow_qb, sc.slow_nb);
    cudaEventRecord(side.ev_done, side.st);
    ppi::count_launch(mc > 0 ? 6 : 5);
    if (stats_dev) {  // this chunk's statistics, once its queued frames are planned too
      cudaStreamWaitEvent(ls, side.ev_done, 0);
      // (per-frame counters only: the checksum was accumulated by the kernels above, sc.xsum)
      stats_kernel<<<stats_grid(cnt), 256, 0, ls>>>(fout, cnt, (unsigned long long *)stats_dev,
                                                    false);
      ppi::count_launch();
    }
    rc = check_launch("plan pipeline");
    phase_mark(pe, 5, ls);
  }
  // join: every pipe waits for its side stream's last kernels, the caller's stream for every pipe
  for (int k = 0; k < pipes && k < ci; k++) {
    cudaStreamWaitEvent(lane_st[k], lane_side[k]->ev_done, 0);
    if (pipes > 1) {
      cudaEventRecord(pp_.done[k], lane_st[k]);
      cudaStreamWaitEvent(st, pp_.done[k], 0);
    }
  }
  if (dbg) {
    std::vector<int32_t> h((size_t)n_chunks * 2 + 8);
    cudaStreamSynchronize(st);
    cudaMemcpy(h.data(), n_base, counters + 32, cudaMemcpyDeviceToHost);
    long a = 0, b = 0;
    for (int64_t i = 0; i < n_chunks; i++) {
      a += h[2 * i];
      b += h[2 * i + 1];
    }
    const int32_t *r = h.data() + 2 * n_chunks;
    std::fprintf(stderr,
                 "pp_plan_batch: %lld frames, queued by k_decide %ld, by k_emit %ld (knots not "
                 "staged %d, operand outside the lean arithmetic %d)\n",
                 (long long)n_frames, a, b, r[1], r[5]);
  }
  if (!caller_scratch) cudaFreeAsync(buf, st);
  if (rc == PP_OK) rc = check_launch("plan pipeline join");
  return rc;
}

extern "C" int pp_set_pipes(int pipes) {
  if (pipes < 0 || pipes > kMaxPipes) return PP_E_RANGE;
  g_pipes_override = pipes;
  return PP_OK;
}

extern "C" int pp_set_phase_timing(int on) {
  g_phase_timing = on != 0;
  return PP_OK;
}

// Sums the per-phase device times (ms) of every pipeline chunk launched since
// the previous call while phase timing was on; synchronises on the last event.
extern "C" int pp_get_phase_ms(double *ms_out, int64_t *chunks_out) {
  if (!ms_out) return PP_E_ARG;
  for (int i = 0; i < kPhases; i++) ms_out[i] = 0;
  int rc = PP_OK;
  std::lock_guard<std::mutex> lk(g_phase_mu);
  for (PhaseEvents &pe : g_phase_events) {
    if (cudaEventSynchronize(pe.ev[kPhases]) != cudaSuccess) rc = PP_E_CUDA;
    for (int i = 0; i < kPhases && rc == PP_OK; i++) {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, pe.ev[i], pe.ev[i + 1]) != cudaSuccess) rc = PP_E_CUDA;
      ms_out[i] += ms;
    }
    g_phase_pool.push_back(pe);
  }
  if (chunks_out) *chunks_out = (int64_t)g_phase_events.size();
  g_phase_events.clear();
  if (rc != PP_OK) check_launch("pp_get_phase_ms");
  return rc;
}

extern "C" int pp_stats_batch(const pp_plans *p, int64_t n_frames, int64_t *stats_dev,
                              void *cuda_stream) {
  if (!p || !stats_dev || n_frames < 0) return PP_E_ARG;
  if (!p->next_x || !p->next_y || !p->n_points || !p->ego_lane || !p->target_lane || !p->flags)
    return PP_E_ARG;
  cudaStream_t st = (cudaStream_t)cuda_stream;
  if (cudaMemsetAsync(stats_dev, 0, PP_STATS_LEN * sizeof(int64_t), st) != cudaSuccess)
    return check_launch("pp_stats_batch memset");
  if (n_frames == 0) return PP_OK;
  stats_kernel<<<stats_grid(n_frames), 256, 0, st>>>(*p, n_frames, (unsigned long long *)stats_dev,
                                                     true);
  ppi::count_launch();
  return check_launch("stats_kernel");
}
