// pp_rollout.cu — closed-loop rollouts (BASELINE config 3): a device-resident
// simulator model around pp_plan_batch.  The model is specified in include/pp.h
// (pp_rollouts); every operation in it is + - * / (and one sqrt) so that the CPU
// restatement the tests check it against is bit-identical.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <utility>
#include <vector>

#include "pp_device.cuh"
#include "pp_internal.h"

namespace {

constexpr int kB = 256;
constexpr double kTick = 0.02;

// splitmix64, as in pp_synth.cpp
__host__ __device__ inline uint64_t mix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
__host__ __device__ inline double u01(uint64_t v) {
  return (double)(v >> 11) * (1.0 / 9007199254740992.0);
}

// The map as the simulator sees it: rows of PP_MAP_STRIDE doubles, index wrapped into [0, n).
struct Track {
  const double *t;  // row 0
  int n;
  int stride;
  __host__ __device__ const double *row(int i) const {
    int k = i;
    if ((unsigned)i >= (unsigned)n) {  // the simulator keeps indices in [0, n): rarely taken
      k = i % n;
      if (k < 0) k += n;
    }
    return t + (size_t)k * stride;
  }
  __host__ __device__ double len(int w, int lane) const { return row(w)[10 + lane]; }
  // walk ds metres along lane `lane` from (w, u)
  __host__ __device__ void walk(int &w, double &u, int lane, double ds) const {
    for (int guard = 0; guard < 4 * n; guard++) {
      const double l = len(w, lane);
      if (ds >= 0) {
        const double rem = l * (1 - u);
        if (ds <= rem) {
          u += ds / l;
          break;
        }
        ds -= rem;
        u = 0;
        w++;
      } else {
        const double rem = l * u;
        if (-ds <= rem) {
          u += ds / l;
          break;
        }
        ds += rem;
        u = 1;
        w--;
      }
    }
    w %= n;
    if (w < 0) w += n;
  }
  // position and unit lane tangent of a car at (lane, w, u)
  __host__ __device__ void pose(int lane, int w, double u, double &x, double &y, double &tx,
                                double &ty) const {
    const double *a = row(w - 1), *b = row(w);
    const double ax = a[2 + 2 * lane], ay = a[3 + 2 * lane];
    const double bx = b[2 + 2 * lane], by = b[3 + 2 * lane];
    const double l = b[10 + lane];
    x = ax + (bx - ax) * u;
    y = ay + (by - ay) * u;
    tx = (bx - ax) / l;
    ty = (by - ay) / l;
  }
  // position and velocity of a car at (lane, w, u) moving at v
  __host__ __device__ void car(int lane, int w, double u, double v, double &x, double &y,
                               double &vx, double &vy) const {
    double tx, ty;
    pose(lane, w, u, x, y, tx, ty);
    vx = v * tx;
    vy = v * ty;
  }
};

// The key of episode e of rollout `rollout` (pp.h, pp_rollouts_set_restart); episode 0's is the
// key pp_rollouts_create draws with.
__host__ __device__ inline uint64_t episode_key(uint64_t seed, int64_t rollout, int64_t e) {
  const uint64_t k0 = mix64(mix64(seed ^ 0x1417ull) ^ ((uint64_t)rollout * 0xD1B54A32D192ED03ull));
  return e == 0 ? k0 : mix64(k0 + (uint64_t)e * 0xA0761D6478BD642Full);
}

// The ego of a draw: at rest at the centre of `lane` on segment w, and its lane direction
// (vx, vy) at unit speed, which the host turns into the yaw.
struct EgoDraw {
  double x, y, vx, vy;
  int lane, w;
};

// One rollout's initial state from its key (pp.h, pp_rollouts_create): the ego, then c cars into
// the rollout's car rows cl / cw / cr / cs.
__host__ __device__ inline EgoDraw draw_rollout(const Track &trk, uint64_t key, int c, int32_t *cl,
                                                int32_t *cw, double *cr, double *cs) {
  uint64_t ctr = 0;
  auto uni = [&]() { return u01(mix64(key + (ctr++) * 0x9E3779B97F4A7C15ull)); };
  EgoDraw eg;
  int w = (int)(uni() * trk.n);
  if (w >= trk.n) w = trk.n - 1;
  const double u = uni();
  int lane = (int)(uni() * 3);
  if (lane > 2) lane = 2;
  trk.car(lane, w, u, 1.0, eg.x, eg.y, eg.vx, eg.vy);
  eg.lane = lane;
  eg.w = w;
  for (int j = 0; j < c; j++) {
    int l = (int)(uni() * 3);
    if (l > 2) l = 2;
    const double ds = -100.0 + 400.0 * uni();
    const double sp = 17.88 + 8.94 * uni();
    int ww = w;
    double uu = u;
    trk.walk(ww, uu, l, ds);
    cl[j] = l;
    cw[j] = ww;
    cr[j] = uu;
    cs[j] = sp;
  }
  return eg;
}

// The ego's yaw from its lane direction, on the host (device atan2 need not give the same bits).
inline double ego_yaw_deg(double vx, double vy) { return std::atan2(vy, vx) * 180 / M_PI; }

// Incident monitor state on the device (definitions: pp.h, pp_rollout_incidents).  Per-rollout
// arrays are indexed by the absolute rollout; [x][R] arrays are row-major in x, so the ego warp's
// lanes (consecutive rollouts) touch consecutive words.
struct Monitor {
  double2 *ring;        // [PP_INC_HISTORY][R]: driven point D_j in row j % PP_INC_HISTORY
  double2 *ring_acc;    // [PP_INC_HISTORY][R]: A_j beside it (0 while undefined)
  int64_t *pts;         // [R] index i of the ego's current point D_i
  uint32_t *active;     // [R] bit per kind: its condition held at the last evaluation
  int32_t *off_pts;     // [R] driven points off the lane centre in a row
  int32_t *count;       // [PP_INC_KINDS][R]
  int64_t *first_tick;  // [R]
  int32_t *first_kind;  // [R]
  double *dist, *clean, *best, *vmax, *amax, *jmax;  // [R]
  const double *ego0_x, *ego0_y;  // [R] the ego before the tick (this tick's frame)
  int64_t R;
};

// State of the IDM traffic model on the device (pp.h, PP_TRAFFIC_IDM).  The ego's lane state is
// double-buffered by the rollout's tick parity: tick t reads copy t % 2 (its pre-tick state) and
// writes copy (t + 1) % 2.
struct Traffic {
  double *v0, *acc;          // [R][C] desired speed, last applied acceleration
  const double *cum;         // [3][n + 1] cum(L, w); Lambda_L = cum[L][n]
  int32_t *ego_lanes;        // [2][R] bit L: the ego leads lane L
  double *ego_s;             // [2][3][R] S_ego per lane
  const double *ego0_mph;    // [R] the ego's speed before the tick (this tick's frame)
  int64_t R;
};

// The flight recorder on the device (pp.h, pp_rollouts_set_recorder).  The ring is W slots of
// R * (25 + 4C) words, each laid out like the frames ([field][R...]), so a slot's stores coalesce
// exactly like the frame stores beside them.  Within a slot, in units of R words: ego_x 0, ego_y 1,
// ego_yaw_deg 2, ego_speed_mph 3, prev_x 4 (x10), prev_y 14 (x10), car_x 24, car_y 24 + C,
// car_vx 24 + 2C, car_vy 24 + 3C (xC each), then prev_n and target_lane_in as int32 [R] each.
struct Recorder {
  double *ring;
  int64_t *trig_tick;   // [R] tick the rollout froze in, -1 while it records
  uint32_t *trig_bits;  // [R]
  int64_t R;
  int c, W;
  unsigned mask;
  __host__ __device__ int64_t slot_words() const { return (int64_t)(25 + 4 * c) * R; }
  __device__ double *slot(int s) const { return ring + s * slot_words(); }
  __device__ int32_t *ints(int s) const { return (int32_t *)(slot(s) + (int64_t)(24 + 4 * c) * R); }
};
static_assert(PP_INC_COLLISION_FRONT == 0 && PP_INC_COLLISION_REAR == 1,
              "k_sim_advance: the collision word's bits are the trigger bits");

// The near-miss record on the device (pp.h, pp_rollouts_set_surrogate).
struct Surrogate {
  double *min;        // [PP_SSM_MEASURES][R]
  int64_t *min_tick;  // [R] tick min_ttc_front was last lowered in
  int32_t *hist;      // [PP_SSM_MEASURES][PP_SSM_BINS][R]
  int64_t R;
};
constexpr unsigned long long kInfBits = 0x7FF0000000000000ull;  // +inf

// The episode-restart mode on the device (pp.h, pp_rollouts_set_restart).
struct Restart {
  int32_t *count0;        // [PP_INC_KINDS][R] the monitor's counts after the last tick
  double *dist0;          // [R] distance_m after the last tick (the restore of a non-finite one)
  int64_t *episodes;      // [R]
  int64_t *by_bit;        // [PP_INC_KINDS + 1][R]
  int64_t *ep_tick;       // [R]
  double *ep_m, *ended_m; // [R]
  int64_t *ended_lap;     // [R]
  const double *yaw;      // [3][n] the ego's yaw at the centre of lane L on segment w (host atan2)
  int64_t R;
  unsigned mask;
};

// Bin of a value >= +0: the number of edges at or below it (PP_SSM_BINS: not counted).
__host__ __device__ inline int ssm_bin(double v) {
  constexpr double e[PP_SSM_BINS] = PP_SSM_EDGES;
  int b = 0;
#pragma unroll
  for (int i = 0; i < PP_SSM_BINS; i++) b += v < e[i] ? 0 : 1;
  return b;
}

// The ego's lane state from its reference and lane match (pp.h, PP_TRAFFIC_IDM).
__device__ __forceinline__ void traffic_ego_state(const Track &trk, const Traffic &tf, int64_t r,
                                                  int buf, const ppd::RefState &rs,
                                                  const ppd::Match &mt) {
  int w = rs.wp % trk.n;
  if (w < 0) w += trk.n;
  int lanes = 0;
#pragma unroll
  for (int L = 0; L < 3; L++) {
    if (mt.ok && fabs(mt.d - (4.0 * L + 2.0)) < PP_TRF_EGO_CORRIDOR) lanes |= 1 << L;
    tf.ego_s[((int64_t)buf * 3 + L) * tf.R + r] = tf.cum[L * (trk.n + 1) + w] + rs.ratio[L] * trk.len(rs.wp, L);
  }
  tf.ego_lanes[buf * tf.R + r] = lanes;
}

// Reduce Delta = S_c - S_f into [0, lam) with at most one addition or subtraction.
__host__ __device__ inline double traffic_delta(double sc, double sf, double lam) {
  double d = sc - sf;
  if (d < 0) {
    d += lam;
  } else if (d >= lam) {
    d -= lam;
  }
  return d;
}

// The IDM acceleration of a car at speed v with desired speed v0 behind a leader Delta ahead at
// speed vl (has_lead false: free road), clamped.
__host__ __device__ inline double traffic_idm_acc(double v, double v0, bool has_lead, double delta,
                                                  double vl) {
  const double q = v / v0, q2 = q * q;
  double inter = 0.0;
  if (has_lead) {
    double gap = delta - PP_INC_CAR_HALF_LEN;
    if (gap < PP_TRF_GAP_FLOOR) gap = PP_TRF_GAP_FLOOR;
    double dyn = v * PP_TRF_HEADWAY + v * (v - vl) / (2.0 * sqrt(PP_TRF_ACC * PP_TRF_DEC));
    if (dyn < 0.0) dyn = 0.0;
    const double s_star = PP_TRF_MIN_GAP + dyn;
    const double z = s_star / gap;
    inter = z * z;
  }
  double acc = PP_TRF_ACC * (1.0 - q2 * q2 - inter);
  if (acc < -PP_TRF_MAX_DEC) acc = -PP_TRF_MAX_DEC;
  if (acc > PP_TRF_ACC) acc = PP_TRF_ACC;
  return acc;
}

// 0 = no overlap, 1 = overlap with the car ahead of the ego along its lane, 2 = any other
__host__ __device__ inline int car_overlap(double cx, double cy, double tx, double ty, double ex,
                                           double ey) {
  const double dx = cx - ex, dy = cy - ey;
  const double along = dx * tx + dy * ty;
  const double across = dx * ty - dy * tx;
  if (!(fabs(along) < PP_INC_CAR_HALF_LEN && fabs(across) < PP_INC_CAR_HALF_WIDTH)) return 0;
  return along > 0 ? 1 : 2;
}

// An incident of `kind` counted at tick t (rare: read-modify-write of the record).
// Out of line, with plain pointer arguments (a Monitor by reference would be copied to the stack).
__device__ __forceinline__ void count_incident(int32_t *count, int64_t *first_tick, int32_t *first_kind,
                                            int64_t R, int64_t r, int kind, int64_t t) {
  count[kind * R + r] += 1;
  if (kind == PP_INC_COLLISION_REAR) return;
  const int64_t ft = first_tick[r];
  if (ft < 0) {
    first_tick[r] = t;
    first_kind[r] = kind;
  } else if (ft == t && kind < first_kind[r]) {
    first_kind[r] = kind;
  }
}
__device__ __forceinline__ void monitor_count(const Monitor &mo, int64_t r, int kind, int64_t t) {
  count_incident(mo.count, mo.first_tick, mo.first_kind, mo.R, r, kind, t);
}

// a / 0.2, correctly rounded like the division it replaces: Markstein's sequence with
// RN(1 / 0.2) = 5 (ppd::div_rcp) on the common path, so the generic division's subroutine, which
// costs this kernel registers and spills, is only reached outside the safe range.  A zero keeps
// its sign.
__device__ __forceinline__ double div02(double a) {
  const bool z = ppd::is_zero(a);
  if (z || ppd::safe_mag(a)) {
    const double q = ppd::div_rcp(a, 0.2, 5.0);
    return z ? a : q;
  }
  return a / 0.2;
}

// The driven points of one tick, a lane per rollout of the ego warp: distance, clean distance,
// Vbar / A / J, their maxima and the edges of over-speed / -acceleration / -jerk.  The rollout
// drove k >= 1 points from (ox, oy) through row nx / ny of the new plan.  Returns the active bits
// with the kinematic ones updated; clean_m is stored, the active bits are left to the caller.
// A_i is kept beside D_i in the history, so J_i reads A_{i-50} instead of recomputing it from
// four points (the same operations on the same values: the same bits, fewer registers).
// kRec: the kinds counted are also OR-ed into `fired` (the recorder's triggers).
template <bool kRec>
__device__ __forceinline__ unsigned monitor_points(const Monitor &mo, int64_t r, int k, double ox,
                                                   double oy, const double *nx, const double *ny,
                                                   unsigned act, int64_t t, unsigned &fired) {
  constexpr int H = PP_INC_HISTORY;
  constexpr unsigned kKin = (1u << PP_INC_OVER_SPEED) | (1u << PP_INC_OVER_ACC) | (1u << PP_INC_OVER_JERK);
  const int64_t R = mo.R;
  int64_t i = mo.pts[r];
  int slot = (int)(i % H);
  double px = ox, py = oy;
  for (int j = 0; j < k; j++) {
    const double x = nx[j], y = ny[j];
    i++;
    slot = slot + 1 == H ? 0 : slot + 1;
    auto row = [&](int b) {  // history row of D_{i-b}, 10 <= b < H
      const int s = slot - b;
      return (int64_t)(s < 0 ? s + H : s) * R + r;
    };
    const double sx = x - px, sy = y - py;
    const double step = sqrt(sx * sx + sy * sy);
    mo.dist[r] += step;
    double clean = mo.clean[r] + step;
    if (clean > mo.best[r]) mo.best[r] = clean;
    unsigned cond = 0;
    double2 acc = make_double2(0.0, 0.0);
    if (i >= 10) {
      const double2 d10 = mo.ring[row(10)];
      const double vx = div02(x - d10.x), vy = div02(y - d10.y);
      const double v = sqrt(vx * vx + vy * vy);
      if (v > mo.vmax[r]) mo.vmax[r] = v;
      if (v > PP_INC_MAX_SPEED) cond |= 1u << PP_INC_OVER_SPEED;
      if (i >= 20) {
        const double2 d20 = mo.ring[row(20)];
        const double wx = div02(d10.x - d20.x), wy = div02(d10.y - d20.y);
        acc.x = div02(vx - wx);
        acc.y = div02(vy - wy);
        const double a = sqrt(acc.x * acc.x + acc.y * acc.y);
        if (a > mo.amax[r]) mo.amax[r] = a;
        if (a > PP_INC_MAX_ACC) cond |= 1u << PP_INC_OVER_ACC;
        if (i >= H) {
          const double2 a50 = mo.ring_acc[row(50)];
          const double jx = (acc.x - a50.x) / 1.0, jy = (acc.y - a50.y) / 1.0;
          const double jn = sqrt(jx * jx + jy * jy);
          if (jn > mo.jmax[r]) mo.jmax[r] = jn;
          if (jn > PP_INC_MAX_JERK) cond |= 1u << PP_INC_OVER_JERK;
        }
      }
    }
    mo.ring[(int64_t)slot * R + r] = make_double2(x, y);
    mo.ring_acc[(int64_t)slot * R + r] = acc;
    const unsigned rise = cond & ~act;
    act = (act & ~kKin) | cond;
    if (rise) {
      for (int kind = PP_INC_OVER_SPEED; kind <= PP_INC_OVER_JERK; kind++)
        if ((rise >> kind) & 1u) monitor_count(mo, r, kind, t);
      clean = 0;
      if constexpr (kRec) fired |= rise;
    }
    mo.clean[r] = clean;
    px = x;
    py = y;
  }
  mo.pts[r] = i;
  return act;
}

// The lateral position of P, a lane per rollout of a whole warp (the lane matching votes across
// it): the reference waypoint from the plan's ref_wp +- 3, then Map::lane_matching.  Keeps the
// off-centre count of a rollout that drove k >= 1 points and returns the out-of-lane / off-road
// condition bits (0 when it drove none).  The reference and the match are left in rs / mt.
__device__ __forceinline__ unsigned monitor_lateral(const Track &trk, const Monitor &mo, int64_t r,
                                                    int k, double px, double py, int ref_wp,
                                                    ppd::RefState &rs, ppd::Match &mt) {
  const ppd::MapView mv{trk.t, trk.n, trk.n < PPD_PAD ? trk.n : PPD_PAD};
  int closest = ref_wp - 3;
  {
    const double *w0 = ppd::row(mv, closest);
    double bd = (w0[0] - px) * (w0[0] - px) + (w0[1] - py) * (w0[1] - py);
    for (int w = ref_wp - 2; w <= ref_wp + 3; w++) {
      const double *rw = ppd::row(mv, w);
      const double d = (rw[0] - px) * (rw[0] - px) + (rw[1] - py) * (rw[1] - py);
      if (d < bd) {
        closest = w;
        bd = d;
      }
    }
  }
  ppd::finish_reference(mv, px, py, closest, rs);
  mt = ppd::lane_match(mv, rs, px, py);
  if (k <= 0) return 0;
  const bool off_centre = !mt.ok || fabs(mt.d - ppd::lane_center_offset(mt.lane)) > PP_INC_LANE_TOL;
  int off = mo.off_pts[r];
  if (!off_centre) {
    off = 0;
  } else if (off < (1 << 30)) {
    off += k;
  }
  mo.off_pts[r] = off;
  unsigned cond = 0;
  if (off > PP_INC_OUT_POINTS) cond |= 1u << PP_INC_OUT_OF_LANE;
  if (!mt.ok || mt.d < PP_INC_ROAD_MIN_D || mt.d > PP_INC_ROAD_MAX_D) cond |= 1u << PP_INC_OFF_ROAD;
  return cond;
}

// Simulator state on the device (per rollout unless noted).  The unconsumed points of the last
// plan are not copied anywhere: they stay in the plan buffer and `path_off` says where they start.
struct SimState {
  double *ego_x, *ego_y, *ego_yaw, *ego_mph;
  int32_t *path_n, *path_off, *target_lane;
  int32_t *car_lane, *car_wp;       // [R][C]
  double *car_ratio, *car_speed;    // [R][C]
  int64_t *ticks;
};

// Both simulator kernels give a block of kB threads only kR rollouts: at 8,192 rollouts per stream
// group a tick is a chain of short dependent kernels, the job is bound by how long ONE frame
// takes to get through that chain (frames in flight / latency), and with a rollout per thread
// these two kernels were 31 and 68 us of it — twelve dependent trips over a thread's car slots,
// fifty over its trajectory row.  Eight threads per rollout make that two trips and seven.
constexpr int kR = 32;  // rollouts per block (one warp's worth: the ego part is one warp)

// One car's near-miss measures against the ego at P = (px, py) moving at U (pp.h), merged into
// the rollout's three shared words.  Every defined value is >= +0, and non-negative doubles order
// like their bits, so an unsigned 64-bit atomicMin is an order-independent minimum.
__device__ __forceinline__ void ssm_car(double cx, double cy, double tx, double ty, double px,
                                        double py, double ux, double uy, double v,
                                        unsigned long long *s_min) {
  const double dx = cx - px, dy = cy - py;
  const double along = dx * tx + dy * ty;
  const double across = dx * ty - dy * tx;
  if (!(fabs(across) < PP_INC_CAR_HALF_WIDTH)) return;
  const double ut = ux * tx + uy * ty;
  if (along >= PP_INC_CAR_HALF_LEN) {
    const double gap = along - PP_INC_CAR_HALF_LEN;
    const double w = ut - v;
    if (w > 0) atomicMin(&s_min[PP_SSM_TTC_FRONT * kR], (unsigned long long)__double_as_longlong(gap / w));
    if (ut > 0) atomicMin(&s_min[PP_SSM_THW * kR], (unsigned long long)__double_as_longlong(gap / ut));
  } else if (along <= -PP_INC_CAR_HALF_LEN) {
    const double gap = -along - PP_INC_CAR_HALF_LEN;
    const double w = v - ut;
    if (w > 0) atomicMin(&s_min[PP_SSM_TTC_REAR * kR], (unsigned long long)__double_as_longlong(gap / w));
  }
}

// The ego warp's merge of a rollout's tick values into its record (rare stores: a minimum is
// lowered, or a value falls below the last edge).
__device__ __forceinline__ void ssm_merge(const Surrogate &sg, int64_t r, int64_t tick, int k,
                                          const unsigned long long *s_min) {
  const int weight = k > 0 ? k : 1;
#pragma unroll
  for (int m = 0; m < PP_SSM_MEASURES; m++) {
    const double v = __longlong_as_double((long long)s_min[m * kR]);
    const int b = ssm_bin(v);
    if (b < PP_SSM_BINS) sg.hist[((int64_t)m * PP_SSM_BINS + b) * sg.R + r] += weight;
    if (v < sg.min[m * sg.R + r]) {
      sg.min[m * sg.R + r] = v;
      if (m == PP_SSM_TTC_FRONT) sg.min_tick[r] = tick;
    }
  }
}

// frame <- state.  The block's threads sweep the rollouts' scalars (a warp per field), their
// kept points and their car slots, all coalesced.
// kRec: the frame also goes to the recorder's slot tick % W of each rollout that is not frozen.
template <bool kRec>
__global__ void __launch_bounds__(kB, 6)
k_sim_frames(Track trk, int64_t lo, int64_t n, int c, SimState st, pp_plans pl, pp_frames fr,
             Recorder rc) {
  const int64_t r0 = lo + (int64_t)blockIdx.x * kR;
  int64_t r_end = r0 + kR;
  if (r_end > lo + n) r_end = lo + n;
  const int nr = (int)(r_end - r0);
  int *s_slot = nullptr;  // kRec: per rollout of the block, its slot, -1 frozen (or past the end)
  if constexpr (kRec) {
    __shared__ int slot_[kR];
    if (threadIdx.x < kR) {
      const int64_t r = r0 + threadIdx.x;
      slot_[threadIdx.x] =
          (int)threadIdx.x < nr && rc.trig_tick[r] < 0 ? (int)(st.ticks[r] % rc.W) : -1;
    }
    __syncthreads();
    s_slot = slot_;
  }
  {  // ego scalars: warp w copies field w
    const int field = threadIdx.x >> 5, rr = threadIdx.x & 31;
    const int64_t r = r0 + rr;
    if (rr < nr) {
      switch (field) {
        case 0: const_cast<double *>(fr.ego_x)[r] = st.ego_x[r]; break;
        case 1: const_cast<double *>(fr.ego_y)[r] = st.ego_y[r]; break;
        case 2: const_cast<double *>(fr.ego_yaw_deg)[r] = st.ego_yaw[r]; break;
        case 3: const_cast<double *>(fr.ego_speed_mph)[r] = st.ego_mph[r]; break;
        case 4: const_cast<int32_t *>(fr.prev_n)[r] = st.path_n[r]; break;
        case 5: const_cast<int32_t *>(fr.target_lane_in)[r] = st.target_lane[r]; break;
        case 6: const_cast<int32_t *>(fr.n_cars)[r] = c; break;
        default: break;
      }
    }
    if constexpr (kRec) {
      const int s = s_slot[rr];
      if (s >= 0 && field < 6) {
        double *const d = rc.slot(s);
        switch (field) {
          case 0: d[r] = st.ego_x[r]; break;
          case 1: d[rc.R + r] = st.ego_y[r]; break;
          case 2: d[2 * rc.R + r] = st.ego_yaw[r]; break;
          case 3: d[3 * rc.R + r] = st.ego_mph[r]; break;
          case 4: rc.ints(s)[r] = st.path_n[r]; break;
          default: rc.ints(s)[rc.R + r] = st.target_lane[r]; break;
        }
      }
    }
  }
  // kept points: the unconsumed points of the last plan, behind path_off
  for (int e = threadIdx.x; e < nr * PP_PREV_KEEP; e += kB) {
    const int rr = e / PP_PREV_KEEP, i = e - rr * PP_PREV_KEEP;
    const int64_t r = r0 + rr;
    const bool have = i < st.path_n[r];
    const int64_t src = r * PP_PATH_LEN + st.path_off[r] + i;
    const double px = have ? pl.next_x[src] : 0.0;
    const_cast<double *>(fr.prev_x)[r0 * PP_PREV_KEEP + e] = px;
    const double py = have ? pl.next_y[src] : 0.0;
    const_cast<double *>(fr.prev_y)[r0 * PP_PREV_KEEP + e] = py;
    if constexpr (kRec) {
      const int s = s_slot[rr];
      if (s >= 0) {
        double *const d = rc.slot(s) + r0 * PP_PREV_KEEP + e;
        d[4 * rc.R] = px;
        d[14 * rc.R] = py;
      }
    }
  }
  for (int64_t q = r0 * c + threadIdx.x; q < r_end * c; q += kB) {
    double x, y, vx, vy;
    trk.car(st.car_lane[q], st.car_wp[q], st.car_ratio[q], st.car_speed[q], x, y, vx, vy);
    const_cast<int32_t *>(fr.car_id)[q] = (int32_t)(q % c);
    const_cast<double *>(fr.car_x)[q] = x;
    const_cast<double *>(fr.car_y)[q] = y;
    const_cast<double *>(fr.car_vx)[q] = vx;
    const_cast<double *>(fr.car_vy)[q] = vy;
    if constexpr (kRec) {
      const int s = s_slot[(int)(q - r0 * c) / c];
      if (s >= 0) {
        double *const d = rc.slot(s) + 24 * rc.R + q;
        const int64_t cr = (int64_t)c * rc.R;
        d[0] = x;
        d[cr] = y;
        d[2 * cr] = vx;
        d[3 * cr] = vy;
      }
    }
  }
}
static_assert(kB >= 7 * 32 && kR == 32, "k_sim_frames: a warp per scalar field, a lane per rollout");

// state <- simulator step(plan), and this tick's contribution to the aggregate statistics
// (definition: pp_stats_batch).  Warp 0 advances the egos, a lane per rollout, while the other
// warps sweep the car slots: the two parts touch different state except for the rollout's tick
// counter, which the respawn of a car reads, so only its increment waits behind the barrier
// (with the ego part after the barrier the block's other seven warps sat in it for 59 % of the
// kernel, profiles/r2_k_sim_advance_ncu.txt).  The counters are taken with warp votes, no
// atomics in shared memory.  The trajectory checksum normally comes from the planning kernels,
// which add it up as they write the points (plan_batch_scratch, xsum_add): re-reading 800 bytes
// per rollout for it was two thirds of this kernel's traffic.  For the single-kernel paths of
// small jobs the block takes it here, over its rollouts' rows (one contiguous run).
//
// The incident monitor (pp.h) rides along without a launch of its own.  Before the barrier the
// ego warp walks the driven points, warp 1 matches the lane of each rollout's last point (in
// parallel: it is the longest dependent chain of the monitor), and the car-slot threads test each
// car against the old and the new ego, OR-ing a bit per rollout into shared memory.  After the
// barrier the ego warp only merges those words into the edge bits (an incident is rare).
//
// kTraffic selects the traffic model (pp.h); the constant-speed instantiation ignores `tf`.
// Under PP_TRAFFIC_IDM the car-slot warps first stage the pre-tick (lane, S, v) of their
// rollouts' cars in dynamic shared memory ([slot][rollout], so the lanes of a warp scanning
// different rollouts read different banks and those of one rollout read the same word) and
// meet at a barrier of their own, while warps 0 and 1 go on; warp 1 also stores the ego's lane
// state for the next tick.
//
// kRec: the ego warp, which knows the kinds it counts in the tick (the kinematic ones in
// monitor_points, the lateral ones and the collisions after the barrier), compares them and the
// finiteness of distance_m against the recorder's mask and freezes the rollout's window.
//
// kSsm: the near-miss measures (pp.h).  The car-slot threads, which hold each advanced car and
// the ego's P and E for the collision test, take every car's measures and atomicMin them into
// three shared words per rollout (set to +inf beside the s_coll clear); after the block barrier
// the ego warp merges the words into the record.
template <int kTraffic, bool kRec, bool kSsm>
__global__ void __launch_bounds__(kB)
k_sim_advance(Track trk, int64_t lo, int64_t n, int c, uint64_t seed, int64_t first, int consume_k,
              SimState st, pp_plans pl, unsigned long long *stats_sum, int do_xsum, Monitor mo,
              Traffic tf, Recorder rc, Surrogate sg) {
  constexpr bool kIdm = kTraffic == PP_TRAFFIC_IDM;
  __shared__ unsigned s_coll[kR];  // per rollout: bit 0 a front, bit 1 a rear collision began
  __shared__ unsigned s_lat[kR];   // per rollout: out-of-lane / off-road condition bits
  unsigned long long *s_ssm = nullptr;  // kSsm: [PP_SSM_MEASURES][kR] bits of the tick's minima
  if constexpr (kSsm) {
    __shared__ unsigned long long ssm_[PP_SSM_MEASURES * kR];
    s_ssm = ssm_;
  }
  const int64_t r0 = lo + (int64_t)blockIdx.x * kR;
  int64_t r_end = r0 + kR;
  if (r_end > lo + n) r_end = lo + n;
  const int nr = (int)(r_end - r0);
  unsigned act = 0, act0 = 0;  // the ego warp's edge bits of its rollout, before and after
  unsigned fired = 0;          // kRec: the kinematic kinds the ego warp counted in this tick
  int64_t tick = 0;
  bool drove = false;
  int k_ssm = 0;  // kSsm: the ego warp's k, kept for the merge after the barrier
  if (threadIdx.x < 32) {
    s_coll[threadIdx.x] = 0;
    if constexpr (kSsm) {
#pragma unroll
      for (int m = 0; m < PP_SSM_MEASURES; m++) s_ssm[m * kR + threadIdx.x] = kInfBits;
    }
    asm volatile("bar.arrive 1, %0;" ::"n"(kB - 32) : "memory");  // the car-slot threads may OR now
    // ---- the ego consumes k points of the new trajectory (one lane per rollout)
    const int ln = threadIdx.x;
    const bool live = ln < nr;
    const int64_t r = r0 + (live ? ln : 0);
    const int np = live ? pl.n_points[r] : 0;
    const int k = live ? (consume_k < np ? consume_k : np) : 0;
    const double ox = st.ego_x[r], oy = st.ego_y[r];
    tick = st.ticks[r];
    act0 = act = mo.active[r];
    drove = k > 0;
    if constexpr (kSsm) k_ssm = k;
    int tl = -1, el = -1;
    uint32_t fl = 0;
    if (live) {
      if (k > 0) {
        const double qx = pl.next_x[r * PP_PATH_LEN + k - 1], qy = pl.next_y[r * PP_PATH_LEN + k - 1];
        const double d = sqrt((qx - ox) * (qx - ox) + (qy - oy) * (qy - oy));
        st.ego_x[r] = qx;
        st.ego_y[r] = qy;
        st.ego_mph[r] = d / (kTick * k) * 2.237;
      }
      st.path_n[r] = np - k;
      st.path_off[r] = k;
      tl = pl.target_lane[r];
      el = pl.ego_lane[r];
      st.target_lane[r] = tl;
      fl = pl.flags[r];
    }
    if (k > 0)
      act = monitor_points<kRec>(mo, r, k, ox, oy, pl.next_x + r * PP_PATH_LEN,
                                 pl.next_y + r * PP_PATH_LEN, act0, tick, fired);
    // counters: lane i ends up holding entry i of the statistics vector
    const unsigned full = 0xffffffffu;
    unsigned long long mine = 0;
    unsigned long long pts = (unsigned long long)np;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) pts += __shfl_xor_sync(full, pts, o);
    const unsigned n_live = __popc(__ballot_sync(full, live));
    if (ln == PP_STAT_FRAMES) mine = n_live;
    if (ln == PP_STAT_POINTS) mine = pts;
#pragma unroll
    for (int q = 0; q < 3; q++) {
      const unsigned a = __popc(__ballot_sync(full, live && tl == q));
      const unsigned b = __popc(__ballot_sync(full, live && el == q));
      if (ln == PP_STAT_TARGET_LANE0 + q) mine = a;
      if (ln == PP_STAT_EGO_LANE0 + q) mine = b;
    }
    {
      const unsigned a = __popc(__ballot_sync(full, live && tl != el));
      if (ln == PP_STAT_LANE_CHANGES) mine = a;
    }
#pragma unroll
    for (int b = 0; b < PP_NUM_FLAGS; b++) {
      const unsigned a = __popc(__ballot_sync(full, (fl >> b) & 1u));
      if (ln == PP_STAT_FLAG0 + b) mine = a;
    }
    if (ln < PP_STATS_LEN && ln != PP_STAT_XSUM && mine) atomicAdd(&stats_sum[ln], mine);
  } else if (threadIdx.x < 64) {
    // ---- lateral position of the ego after its k points (one lane per rollout)
    const int ln = threadIdx.x - 32;
    const bool live = ln < nr;
    const int64_t r = r0 + (live ? ln : 0);
    const int np = pl.n_points[r];
    const int k = live ? (consume_k < np ? consume_k : np) : 0;
    const double px = k > 0 ? pl.next_x[r * PP_PATH_LEN + k - 1] : mo.ego0_x[r];
    const double py = k > 0 ? pl.next_y[r * PP_PATH_LEN + k - 1] : mo.ego0_y[r];
    ppd::RefState rs;
    ppd::Match mt;
    s_lat[ln] = monitor_lateral(trk, mo, r, k, px, py, pl.ref_wp[r], rs, mt);
    if constexpr (kIdm) {
      if (live) traffic_ego_state(trk, tf, r, (int)((st.ticks[r] + 1) & 1), rs, mt);
    }
  } else {
    asm volatile("bar.sync 1, %0;" ::"n"(kB - 32) : "memory");  // s_coll is cleared
    extern __shared__ double s_trf[];  // IDM: S [c][kR], v [c][kR], then lane [c][kR] (int)
    double *const s_S = s_trf, *const s_v = s_trf + c * kR;
    int *const s_ln = (int *)(s_trf + 2 * c * kR);
    if constexpr (kIdm) {  // ---- stage the cars before the tick
      for (int b = threadIdx.x - 64; b < nr * c; b += kB - 64) {  // b: car slot of the block
        const int rr = b / c, j = b - rr * c, e = j * kR + rr;
        const int64_t q = r0 * c + b;
        const int lane = st.car_lane[q], w = st.car_wp[q];
        s_S[e] = tf.cum[lane * (trk.n + 1) + w] + st.car_ratio[q] * trk.len(w, lane);
        s_v[e] = st.car_speed[q];
        s_ln[e] = lane;
      }
      asm volatile("bar.sync 2, %0;" ::"n"(kB - 64) : "memory");  // the car-slot warps only
      // ---- every car's acceleration from its leader, stored to tf.acc for the advance below
      // (a pass of its own: the scan's registers are free again when the advance runs)
      for (int b = threadIdx.x - 64; b < nr * c; b += kB - 64) {
        const int rr = b / c, j = b - rr * c;
        const int64_t q = r0 * c + b, r = r0 + rr;
        const int lane = s_ln[j * kR + rr];
        const double sf = s_S[j * kR + rr];
        const double lam = tf.cum[lane * (trk.n + 1) + trk.n], half = lam / 2;
        bool has = false;
        double best = 0.0, vl = 0.0;
        for (int i = 0; i < c; i++) {
          if (s_ln[i * kR + rr] != lane) continue;
          const double d = traffic_delta(s_S[i * kR + rr], sf, lam);
          if (((d > 0 && d < half) || (d == 0 && i > j)) && (!has || d < best)) {
            has = true;
            best = d;
            vl = s_v[i * kR + rr];
          }
        }
        const int par = (int)(st.ticks[r] & 1);
        if ((tf.ego_lanes[par * tf.R + r] >> lane) & 1) {
          const double d = traffic_delta(tf.ego_s[((int64_t)par * 3 + lane) * tf.R + r], sf, lam);
          if (((d > 0 && d < half) || d == 0) && (!has || d < best)) {
            has = true;
            best = d;
            vl = tf.ego0_mph[r] / 2.237;
          }
        }
        tf.acc[q] = traffic_idm_acc(s_v[j * kR + rr], tf.v0[q], has, best, vl);
      }
    }
    // ---- traffic (one thread per car slot; they read the rollout's tick before it is counted)
    for (int64_t q = r0 * c + (threadIdx.x - 64); q < r_end * c; q += kB - 64) {
      const int64_t r = q / c;
      const int j = (int)(q - r * c);
      const int np = pl.n_points[r];
      const int k = consume_k < np ? consume_k : np;
      const double dt = kTick * (k > 0 ? k : 1);
      int lane = st.car_lane[q], w = st.car_wp[q];
      double u = st.car_ratio[q], v = st.car_speed[q];
      int was;  // overlap of the car before its advance with the ego before the tick
      {
        double cx, cy, tx, ty;
        trk.pose(lane, w, u, cx, cy, tx, ty);
        was = car_overlap(cx, cy, tx, ty, mo.ego0_x[r], mo.ego0_y[r]);
      }
      const int m_lane = pl.car_lane[q];
      const double m_s = pl.car_s[q];
      if (m_lane < 0 || m_s < -100.0 || m_s > 300.0) {  // respawn
        const int64_t tick = st.ticks[r];
        const uint64_t key = mix64(mix64(seed ^ 0x5157ull) ^ ((uint64_t)(first + r) * 0xD1B54A32D192ED03ull));
        const uint64_t h = mix64(key ^ ((uint64_t)tick * 0x9E3779B97F4A7C15ull) ^ ((uint64_t)j << 48));
        const double u1 = u01(mix64(h + 1)), u2 = u01(mix64(h + 2)), u3 = u01(mix64(h + 3));
        const double ds = (m_lane >= 0 && m_s < -100.0) ? 200.0 + 100.0 * u1 : -(60.0 + 40.0 * u1);
        lane = (int)(3.0 * u2);
        if (lane > 2) lane = 2;
        v = 17.88 + 8.94 * u3;
        w = pl.ref_wp[r];
        u = 0.5;
        trk.walk(w, u, lane, ds);
        if constexpr (kIdm) {
          tf.v0[q] = v;
          tf.acc[q] = 0.0;
        }
      } else if constexpr (kIdm) {  // the IDM step with the acceleration of the pass above
        const double acc = tf.acc[q];
        double v1 = v + acc * dt;
        if (v1 < 0) v1 = 0;
        const double ds = (v + v1) * 0.5 * dt;
        u += ds / trk.len(w, lane);
        for (int guard = 0; guard < 64 && u >= 1; guard++) {
          const double left = (u - 1) * trk.len(w, lane);
          w = w + 1 == trk.n ? 0 : w + 1;
          u = left / trk.len(w, lane);
        }
        v = v1;
      } else {  // constant speed along the lane centre line
        u += (v * dt) / trk.len(w, lane);
        for (int guard = 0; guard < 64 && u >= 1; guard++) {
          const double left = (u - 1) * trk.len(w, lane);
          w = w + 1 == trk.n ? 0 : w + 1;
          u = left / trk.len(w, lane);
        }
      }
      st.car_lane[q] = lane;
      st.car_wp[q] = w;
      st.car_ratio[q] = u;
      st.car_speed[q] = v;
      {  // the same pair now: the car advanced, the ego at its last driven point
        double cx, cy, tx, ty;
        trk.pose(lane, w, u, cx, cy, tx, ty);
        const double ex = k > 0 ? pl.next_x[r * PP_PATH_LEN + k - 1] : mo.ego0_x[r];
        const double ey = k > 0 ? pl.next_y[r * PP_PATH_LEN + k - 1] : mo.ego0_y[r];
        const int now = car_overlap(cx, cy, tx, ty, ex, ey);
        if (now && !was) atomicOr(&s_coll[r - r0], (unsigned)now);
        if constexpr (kSsm) {
          double ux = 0.0, uy = 0.0;
          if (k > 0) {
            ux = (ex - mo.ego0_x[r]) * 50.0 / k;
            uy = (ey - mo.ego0_y[r]) * 50.0 / k;
          }
          ssm_car(cx, cy, tx, ty, ex, ey, ux, uy, v, s_ssm + (r - r0));
        }
      }
    }
  }
  if (do_xsum) {  // ---- checksum of the block's rows, unless the planning kernels added it
    long long xs = 0;
    const int64_t base = r0 * PP_PATH_LEN;
    for (int e = threadIdx.x; e < nr * PP_PATH_LEN; e += kB) {
      const int rr = e / PP_PATH_LEN;
      const int np_r = pl.n_points[r0 + rr];
      const double x = pl.next_x[base + e], y = pl.next_y[base + e];
      if (e - rr * PP_PATH_LEN < np_r && x == x && y == y && fabs(x) < 1e12 && fabs(y) < 1e12)
        xs += (long long)(x * 256.0) + (long long)(y * 256.0);
    }
    unsigned long long v = (unsigned long long)xs;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(&stats_sum[PP_STAT_XSUM], v);
  }
  __syncthreads();
  if (threadIdx.x < nr) {  // the ego warp: lateral edges, then collisions
    const int64_t r = r0 + threadIdx.x;
    constexpr unsigned kLat = (1u << PP_INC_OUT_OF_LANE) | (1u << PP_INC_OFF_ROAD);
    const unsigned cb = s_coll[threadIdx.x];
    if (drove) act = (act & ~kLat) | s_lat[threadIdx.x];
    const unsigned rise = act & ~act0 & kLat;
    if (act != act0) mo.active[r] = act;
    if (rise | cb) {
      for (int kind = PP_INC_OUT_OF_LANE; kind <= PP_INC_OFF_ROAD; kind++)
        if ((rise >> kind) & 1u) monitor_count(mo, r, kind, tick);
      if (cb & 1u) monitor_count(mo, r, PP_INC_COLLISION_FRONT, tick);
      if (cb & 2u) monitor_count(mo, r, PP_INC_COLLISION_REAR, tick);
      if (rise | (cb & 1u)) mo.clean[r] = 0;
    }
    if constexpr (kRec) {
      unsigned hit = fired | rise | cb;
      if (!isfinite(mo.dist[r])) hit |= 1u << PP_REC_NONFINITE;
      hit &= rc.mask;
      if (hit && rc.trig_tick[r] < 0) {
        rc.trig_tick[r] = tick;
        rc.trig_bits[r] = hit;
      }
    }
    if constexpr (kSsm) ssm_merge(sg, r, tick, k_ssm, s_ssm + threadIdx.x);
    st.ticks[r] += 1;
  }
}

// pp_rollouts_incident_totals: counts per kind, rollouts with an incident, millimetres driven.
__global__ void __launch_bounds__(kB) k_incident_totals(Monitor mo, unsigned long long *tot) {
  unsigned long long acc[PP_INC_TOTALS_LEN];
#pragma unroll
  for (int e = 0; e < PP_INC_TOTALS_LEN; e++) acc[e] = 0;
  for (int64_t r = (int64_t)blockIdx.x * kB + threadIdx.x; r < mo.R; r += (int64_t)gridDim.x * kB) {
#pragma unroll
    for (int e = 0; e < PP_INC_KINDS; e++) acc[e] += (unsigned long long)mo.count[e * mo.R + r];
    acc[PP_INC_TOTAL_ROLLOUTS] += mo.first_tick[r] >= 0 ? 1u : 0u;
    acc[PP_INC_TOTAL_MM] += (unsigned long long)llround(mo.dist[r] * 1000.0);
  }
#pragma unroll
  for (int e = 0; e < PP_INC_TOTALS_LEN; e++) {
    unsigned long long v = acc[e];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(&tot[e], v);
  }
}
static_assert(PP_STATS_LEN <= 32, "k_sim_advance: a lane per statistics entry");

// pp_rollouts_surrogate_totals: the histograms summed over the rollouts, then the rollouts per
// bin of their minima.
__global__ void __launch_bounds__(kB) k_surrogate_totals(Surrogate sg, unsigned long long *tot) {
  constexpr int MB = PP_SSM_MEASURES * PP_SSM_BINS;
  unsigned long long acc[PP_SSM_TOTALS_LEN];
#pragma unroll
  for (int e = 0; e < PP_SSM_TOTALS_LEN; e++) acc[e] = 0;
  for (int64_t r = (int64_t)blockIdx.x * kB + threadIdx.x; r < sg.R; r += (int64_t)gridDim.x * kB) {
#pragma unroll
    for (int e = 0; e < MB; e++) acc[e] += (unsigned long long)sg.hist[e * sg.R + r];
#pragma unroll
    for (int m = 0; m < PP_SSM_MEASURES; m++) {
      const int b = ssm_bin(sg.min[m * sg.R + r]);
#pragma unroll
      for (int i = 0; i < PP_SSM_BINS; i++) acc[MB + m * PP_SSM_BINS + i] += b == i ? 1u : 0u;
    }
  }
#pragma unroll
  for (int e = 0; e < PP_SSM_TOTALS_LEN; e++) {
    unsigned long long v = acc[e];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(&tot[e], v);
  }
}
static_assert(PP_SSM_TOTAL_MIN == PP_SSM_MEASURES * PP_SSM_BINS, "k_surrogate_totals: layout");

// The ego's lane state before the first tick (pp.h, PP_TRAFFIC_IDM): the full reference search
// of Map::init_reference_waypoint at the initial pose, then the lane match.  Whole warps run the
// match (it votes across the warp); lanes past the end repeat the last rollout and store nothing.
__global__ void __launch_bounds__(kB) k_traffic_init(Track trk, const double *ex, const double *ey,
                                                     Traffic tf) {
  const int64_t i = (int64_t)blockIdx.x * kB + threadIdx.x;
  const int64_t r = i < tf.R ? i : tf.R - 1;
  const ppd::MapView mv{trk.t, trk.n, trk.n < PPD_PAD ? trk.n : PPD_PAD};
  ppd::RefState rs;
  ppd::init_reference(mv, ex[r], ey[r], rs);
  const ppd::Match mt = ppd::lane_match(mv, rs, ex[r], ey[r]);
  if (i < tf.R) traffic_ego_state(trk, tf, r, 0, rs, mt);
}

// The episode restarts of rollouts lo .. lo+n-1 at the end of a tick (pp.h,
// pp_rollouts_set_restart), a thread per rollout, after k_sim_advance has counted the tick.  The
// fired bits are the kinds whose count rose since the last tick and a non-finite distance_m.
// Restarts are rare, so a restarting thread draws its c cars serially; under IDM it also runs
// k_traffic_init's search at the new pose (lane_match votes among the lanes that enter it).
template <int kTraffic>
__global__ void __launch_bounds__(kB) k_restart(Track trk, int64_t lo, int64_t n, int c,
                                                uint64_t seed, int64_t first, SimState st,
                                                Monitor mo, Traffic tf, Restart rt) {
  const int64_t i = (int64_t)blockIdx.x * kB + threadIdx.x;
  if (i >= n) return;
  const int64_t r = lo + i, R = rt.R;
  unsigned fired = 0;
#pragma unroll
  for (int kind = 0; kind < PP_INC_KINDS; kind++) {
    const int32_t now = mo.count[kind * R + r];
    if (now != rt.count0[kind * R + r]) {
      fired |= 1u << kind;
      rt.count0[kind * R + r] = now;
    }
  }
  double d = mo.dist[r];
  if (!isfinite(d)) fired |= 1u << PP_REC_NONFINITE;
  const unsigned hit = fired & rt.mask;
  if (!hit) {
    rt.dist0[r] = d;
    return;
  }
  if (!isfinite(d)) {
    d = rt.dist0[r];
    mo.dist[r] = d;
  }
  const double ended = d - rt.ep_m[r];
  rt.ended_m[r] += ended;
  if (ended >= PP_RST_RUBRIC_M) rt.ended_lap[r] += 1;
  rt.by_bit[(__ffs(hit) - 1) * R + r] += 1;
  const int64_t e = rt.episodes[r] + 1;
  rt.episodes[r] = e;
  const int64_t tick = st.ticks[r];  // t + 1
  rt.ep_tick[r] = tick;
  rt.ep_m[r] = d;
  rt.dist0[r] = d;
  const int64_t q = r * c;
  const EgoDraw eg = draw_rollout(trk, episode_key(seed, first + r, e), c, st.car_lane + q,
                                  st.car_wp + q, st.car_ratio + q, st.car_speed + q);
  st.ego_x[r] = eg.x;
  st.ego_y[r] = eg.y;
  st.ego_yaw[r] = rt.yaw[eg.lane * trk.n + eg.w];
  st.ego_mph[r] = 0.0;
  st.path_n[r] = 0;
  st.path_off[r] = 0;
  st.target_lane[r] = eg.lane;
  mo.ring[r] = make_double2(eg.x, eg.y);  // D_0 in row 0
  mo.ring_acc[r] = make_double2(0.0, 0.0);
  mo.pts[r] = 0;
  mo.active[r] = 0;
  mo.off_pts[r] = 0;
  mo.clean[r] = 0.0;
  if constexpr (kTraffic == PP_TRAFFIC_IDM) {
    for (int j = 0; j < c; j++) {
      tf.v0[q + j] = st.car_speed[q + j];
      tf.acc[q + j] = 0.0;
    }
    const ppd::MapView mv{trk.t, trk.n, trk.n < PPD_PAD ? trk.n : PPD_PAD};
    ppd::RefState rs;
    ppd::init_reference(mv, eg.x, eg.y, rs);
    const ppd::Match mt = ppd::lane_match(mv, rs, eg.x, eg.y);
    traffic_ego_state(trk, tf, r, (int)(tick & 1), rs, mt);
  }
}

// pp_rollouts_restart_totals: restarts per ending bit, ended laps, ended millimetres.
__global__ void __launch_bounds__(kB) k_restart_totals(Restart rt, unsigned long long *tot) {
  unsigned long long acc[PP_RST_TOTALS_LEN];
#pragma unroll
  for (int e = 0; e < PP_RST_TOTALS_LEN; e++) acc[e] = 0;
  for (int64_t r = (int64_t)blockIdx.x * kB + threadIdx.x; r < rt.R; r += (int64_t)gridDim.x * kB) {
#pragma unroll
    for (int b = 0; b <= PP_INC_KINDS; b++) acc[b] += (unsigned long long)rt.by_bit[b * rt.R + r];
    acc[PP_RST_TOTAL_LAPS] += (unsigned long long)rt.ended_lap[r];
    acc[PP_RST_TOTAL_MM] += (unsigned long long)llround(rt.ended_m[r] * 1000.0);
  }
#pragma unroll
  for (int e = 0; e < PP_RST_TOTALS_LEN; e++) {
    unsigned long long v = acc[e];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(&tot[e], v);
  }
}

// The staging buffer of pp_rollouts_get_recording: m rows of W frames in pp_frames layout (frame
// (i, j) at i * W + j), then the trigger arrays of the m rows.
struct RecOut {
  double *d[10];  // ego_x, ego_y, ego_yaw_deg, ego_speed_mph, prev_x, prev_y, car_x, car_y, car_vx, car_vy
  int32_t *i[2];  // prev_n, target_lane_in
  int64_t *trig_tick;
  uint32_t *trig_bits;
};

// Gathers the windows of m rollouts (rows[i], or i when rows is NULL), oldest frame first: row i
// ends at its trigger tick, or at tick ticks_done - 1 when it is not frozen, and holds its last
// min(end + 1, W) ticks; the slots after those are 0.  blockIdx.y is the field: 0 the trigger
// arrays, 1..12 the frame fields in the order of RecOut.
__global__ void __launch_bounds__(kB) k_rec_gather(Recorder rc, const int64_t *rows, int64_t m,
                                                   int64_t ticks_done, RecOut out) {
  const int fld = blockIdx.y;
  const int W = rc.W, c = rc.c;
  if (fld == 0) {
    for (int64_t i = (int64_t)blockIdx.x * kB + threadIdx.x; i < m; i += (int64_t)gridDim.x * kB) {
      const int64_t r = rows ? rows[i] : i;
      out.trig_tick[i] = rc.trig_tick[r];
      out.trig_bits[i] = rc.trig_bits[r];
    }
    return;
  }
  // words per frame and offset in a slot (units of R words) of the frame field
  const int f = fld - 1;
  const int inner = f == 4 || f == 5 ? PP_PREV_KEEP : (f >= 6 && f < 10 ? c : 1);
  const int64_t off = f < 4 ? f : (f < 6 ? 4 + 10 * (f - 4) : 24 + (int64_t)c * (f - 6));
  // the destination, picked by a switch: indexing the parameter's arrays by a runtime field
  // number would copy RecOut to the stack
  double *dd = nullptr;
  int32_t *di = nullptr;
  switch (f) {
    case 0: dd = out.d[0]; break;
    case 1: dd = out.d[1]; break;
    case 2: dd = out.d[2]; break;
    case 3: dd = out.d[3]; break;
    case 4: dd = out.d[4]; break;
    case 5: dd = out.d[5]; break;
    case 6: dd = out.d[6]; break;
    case 7: dd = out.d[7]; break;
    case 8: dd = out.d[8]; break;
    case 9: dd = out.d[9]; break;
    case 10: di = out.i[0]; break;
    default: di = out.i[1]; break;
  }
  const int64_t total = m * W * inner;
  for (int64_t e = (int64_t)blockIdx.x * kB + threadIdx.x; e < total; e += (int64_t)gridDim.x * kB) {
    const int64_t fi = e / inner, i = fi / W;
    const int k = (int)(e - fi * inner), j = (int)(fi - i * W);
    const int64_t r = rows ? rows[i] : i;
    const int64_t tt = rc.trig_tick[r], end = tt >= 0 ? tt : ticks_done - 1;
    const int64_t filled = end + 1 < W ? end + 1 : W;
    const int s = j < filled ? (int)((end - filled + 1 + j) % W) : -1;
    if (dd) {
      dd[e] = s >= 0 ? rc.slot(s)[off * rc.R + r * inner + k] : 0.0;
    } else {
      di[e] = s >= 0 ? rc.ints(s)[(f - 10) * rc.R + r] : 0;
    }
  }
}

int cuda_fail(const char *what, cudaError_t e) {
  ppi::set_cuda_error(what, (int)e, cudaGetErrorString(e));
  cudaGetLastError();
  return PP_E_CUDA;
}

// Blocking copies of the getters and of pp_rollouts_create's upload.  A null destination or an
// empty copy is skipped; after the first CUDA error nothing more is copied and `e` keeps it.
struct Copy {
  cudaMemcpyKind kind;
  cudaError_t e = cudaSuccess;
  void operator()(void *dst, const void *src, size_t bytes) {
    if (e == cudaSuccess && dst && bytes) e = cudaMemcpy(dst, src, bytes, kind);
  }
  // [K][R] on the device -> [R][K] for the caller
  template <class T>
  void transpose(T *dst, const T *src, size_t R, size_t K) {
    if (!dst) return;
    std::vector<T> t(R * K);
    (*this)(t.data(), src, R * K * sizeof(T));
    for (size_t i = 0; i < R; i++)
      for (size_t k = 0; k < K; k++) dst[i * K + k] = t[k * R + i];
  }
};

}  // namespace

struct pp_rollouts {
  const pp_map *map = nullptr;
  int64_t n = 0;   // rollouts
  int32_t c = 0;   // cars per rollout
  uint64_t seed = 0;
  int64_t first = 0;
  int64_t tick = 0;
  // one device allocation (rollouts_layout): the simulator state, the per-tick frames and plans,
  // the statistics and the incident monitor
  char *buf = nullptr;
  SimState st;
  bool lean = false;  // plans without the per-frame diagnostics and unused per-car outputs
  pp_plans full_pl;   // the complete set of output pointers (restored when lean is switched off)
  // per-tick frames and plans
  pp_frames fr;
  pp_plans pl;
  int64_t *stats_sum;  // running sum of the per-tick statistics over all ticks
  // Rollouts are independent, so they are cut into kGroups ranges that tick on their own
  // streams: one group's short kernels and side-stream tail overlap the other groups' work.
  static constexpr int kGroups = 8;  // streams that exist; PP_ROLLOUT_GROUPS of them are used
  cudaStream_t gs[kGroups] = {};
  cudaEvent_t g_done[kGroups] = {};
  cudaEvent_t fork = nullptr;
  cudaStream_t origin = nullptr;  // graph capture / replay stream (the caller's may be the
                                  // legacy default stream, which cannot be captured)
  cudaEvent_t o_fork = nullptr, o_join = nullptr;
  char *scratch[kGroups] = {};  // the planning pipeline's scratch, one per group
  // one tick of every group, captured once and replayed (a tick is ~50 small launches)
  cudaGraphExec_t graph = nullptr;
  int32_t graph_k = 0;
  pp_config graph_cfg;
  int64_t launches_per_tick = 0;
  int groups_wanted = 0;  // pp_rollouts_set_groups: 0 = automatic
  Monitor mo;  // incident monitor (pp.h, pp_rollout_incidents), in `buf`
  // Each observer below owns one allocation of its own, made only when it is switched on; its
  // view's pointers are null until then.
  int traffic = PP_TRAFFIC_CONSTANT;  // traffic model (pp.h, pp_rollouts_set_traffic)
  char *tf_buf = nullptr;             // the IDM state
  Traffic tf;
  char *rc_buf = nullptr;  // flight recorder (pp.h, pp_rollouts_set_recorder): on while rc.W > 0
  Recorder rc;
  // (first tick, consume_k) of every stretch of ticks run with one consume_k.  All rollouts tick
  // together, so the host knows each tick's k; a window frozen long ago still finds its k here.
  std::vector<std::pair<int64_t, int32_t>> rec_k;
  char *sg_buf = nullptr;  // near-miss measures (pp.h, pp_rollouts_set_surrogate): on while allocated
  Surrogate sg;
  char *rt_buf = nullptr;  // episode restarts (pp.h, pp_rollouts_set_restart): on while allocated
  Restart rt;
};

namespace {

// The layout of pp_rollouts::buf (ppi::Carve).  Plans get all outputs: tests compare them tick by
// tick.
size_t rollouts_layout(pp_rollouts *r, char *base) {
  const size_t N = (size_t)r->n, NC = (size_t)r->n * (size_t)(r->c > 0 ? r->c : 1);
  ppi::Carve cv(base);
  SimState &s = r->st;
  cv.take(s.ego_x, N);
  cv.take(s.ego_y, N);
  cv.take(s.ego_yaw, N);
  cv.take(s.ego_mph, N);
  cv.take(s.path_n, N);
  cv.take(s.path_off, N);
  cv.take(s.target_lane, N);
  cv.take(s.car_lane, NC);
  cv.take(s.car_wp, NC);
  cv.take(s.car_ratio, NC);
  cv.take(s.car_speed, NC);
  pp_frames &f = r->fr;
  cv.take(f.ego_x, N);
  cv.take(f.ego_y, N);
  cv.take(f.ego_yaw_deg, N);
  cv.take(f.ego_speed_mph, N);
  cv.take(f.prev_n, N);
  cv.take(f.prev_x, N * PP_PREV_KEEP);
  cv.take(f.prev_y, N * PP_PREV_KEEP);
  cv.take(f.target_lane_in, N);
  cv.take(f.n_cars, N);
  cv.take(f.car_id, NC);
  cv.take(f.car_x, NC);
  cv.take(f.car_y, NC);
  cv.take(f.car_vx, NC);
  cv.take(f.car_vy, NC);
  pp_plans &p = r->pl;
  cv.take(p.next_x, N * PP_PATH_LEN);
  cv.take(p.next_y, N * PP_PATH_LEN);
  cv.take(p.n_points, N);
  cv.take(p.ego_lane, N);
  cv.take(p.ref_wp, N);
  cv.take(p.target_lane, N);
  cv.take(p.flags, N);
  cv.take(p.ego_s, N);
  cv.take(p.ego_d, N);
  cv.take(p.ego_vs, N);
  cv.take(p.ego_vd, N);
  cv.take(p.ego_speed, N);
  cv.take(p.ego_acc, N);
  cv.take(p.target_speed, N);
  cv.take(p.target_time, N);
  cv.take(p.next_car_id, N);
  cv.take(p.next_car_in_target_lane, N);
  cv.take(p.car_s, NC);
  cv.take(p.car_d, NC);
  cv.take(p.car_vs, NC);
  cv.take(p.car_vd, NC);
  cv.take(p.car_lane, NC);
  cv.take(p.car_next_wp, NC);
  cv.take(r->stats_sum, PP_STATS_LEN);
  cv.take(s.ticks, N);
  Monitor &m = r->mo;
  cv.take(m.ring, N * PP_INC_HISTORY);
  cv.take(m.ring_acc, N * PP_INC_HISTORY);
  cv.take(m.pts, N);
  cv.take(m.first_tick, N);
  cv.take(m.active, N);
  cv.take(m.off_pts, N);
  cv.take(m.count, N * PP_INC_KINDS);
  cv.take(m.first_kind, N);
  for (double **d : {&m.dist, &m.clean, &m.best, &m.vmax, &m.amax, &m.jmax}) cv.take(*d, N);
  return cv.size;
}

// An observer's own block for `layout`, a ppi::Carve layout that binds the observer's view and
// returns its size.  The block stays null when the allocation fails.
template <class Layout>
cudaError_t observer_alloc(char *&block, Layout layout) {
  const cudaError_t e = cudaMalloc((void **)&block, layout(nullptr));
  if (e != cudaSuccess) {
    block = nullptr;
    return e;
  }
  layout(block);
  return cudaSuccess;
}

// Frees an observer's block; its layout run without a base leaves the view's pointers null.
template <class Layout>
void observer_free(char *&block, Layout layout) {
  cudaFree(block);
  block = nullptr;
  layout(nullptr);
}

// The totals entry points: zero `len` totals on the caller's stream, then `kernel` adds every
// rollout's record into them.
template <class View>
int record_totals(const pp_rollouts *r, const char *who, void (*kernel)(View, unsigned long long *),
                  const char *kernel_name, const View &view, int len, int64_t *totals_dev,
                  void *cuda_stream) {
  const int rc = ppi::check_map_device(r->map, who);
  if (rc != PP_OK) return rc;
  cudaStream_t st = (cudaStream_t)cuda_stream;
  cudaError_t e = cudaMemsetAsync(totals_dev, 0, len * sizeof(int64_t), st);
  if (e != cudaSuccess) return cuda_fail(who, e);
  const int64_t blocks = (r->n + kB - 1) / kB;
  kernel<<<(int)(blocks < 1184 ? blocks : 1184), kB, 0, st>>>(view, (unsigned long long *)totals_dev);
  ppi::count_launch(1);
  e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(kernel_name, e);
  return PP_OK;
}


}  // namespace

extern "C" int pp_rollouts_create(const pp_map *map, int64_t n, int32_t c, uint64_t seed,
                                  int64_t first, pp_rollouts **out) {
  if (!out) return PP_E_ARG;
  *out = nullptr;
  if (!map || n <= 0 || c < 0 || c > PP_MAX_CARS) return PP_E_ARG;
  {
    const int rc = ppi::check_map_device(map, "pp_rollouts_create");
    if (rc != PP_OK) return rc;
  }
  pp_rollouts *r = new (std::nothrow) pp_rollouts();
  if (!r) return PP_E_NOMEM;
  r->map = map;
  r->n = n;
  r->c = c;
  r->seed = seed;
  r->first = first;
  const size_t N = (size_t)n, NC = (size_t)n * (size_t)(c > 0 ? c : 1);
  const size_t bytes = rollouts_layout(r, nullptr);
  cudaError_t e = cudaMalloc((void **)&r->buf, bytes);
  if (e != cudaSuccess) {
    delete r;
    return cuda_fail("cudaMalloc(rollouts)", e);
  }
  cudaMemset(r->buf, 0, bytes);
  rollouts_layout(r, r->buf);
  r->fr.max_cars = c > 0 ? c : 1;
  r->fr.reserved = 0;
  r->mo.ego0_x = r->fr.ego_x;
  r->mo.ego0_y = r->fr.ego_y;
  r->mo.R = n;
  r->tf = Traffic{nullptr, nullptr, nullptr, nullptr, nullptr, r->fr.ego_speed_mph, n};
  r->rc = Recorder{nullptr, nullptr, nullptr, n, c, 0, 0};
  r->sg = Surrogate{nullptr, nullptr, nullptr, n};
  r->rt = Restart{};
  r->rt.R = n;
  cudaMemset(r->mo.first_tick, 0xff, N * 8);  // -1: no incident yet
  cudaMemset(r->mo.first_kind, 0xff, N * 4);

  // ---- initial state on the host: a pure function of (seed, first + r)
  std::vector<double> ex(N), ey(N), yaw(N), mph(N), cr(NC), cs(NC);
  std::vector<int32_t> tl(N), cl(NC), cw(NC);
  Track trk{map->table.data(), map->n, PP_MAP_STRIDE};
  for (int64_t i = 0; i < n; i++) {
    const size_t q = (size_t)i * c;
    const EgoDraw eg = draw_rollout(trk, episode_key(seed, first + i, 0), c, cl.data() + q,
                                    cw.data() + q, cr.data() + q, cs.data() + q);
    ex[i] = eg.x;
    ey[i] = eg.y;
    yaw[i] = ego_yaw_deg(eg.vx, eg.vy);
    mph[i] = 0.0;
    tl[i] = eg.lane;
  }
  Copy up{cudaMemcpyHostToDevice};
  up(r->st.ego_x, ex.data(), N * 8);
  up(r->st.ego_y, ey.data(), N * 8);
  up(r->st.ego_yaw, yaw.data(), N * 8);
  up(r->st.ego_mph, mph.data(), N * 8);
  up(r->st.target_lane, tl.data(), N * 4);
  {  // D_0, the initial pose, in row 0 of the monitor's history
    std::vector<double> d0(2 * N);
    for (size_t i = 0; i < N; i++) {
      d0[2 * i] = ex[i];
      d0[2 * i + 1] = ey[i];
    }
    up(r->mo.ring, d0.data(), N * 16);
  }
  if (c > 0) {
    up(r->st.car_lane, cl.data(), NC * 4);
    up(r->st.car_wp, cw.data(), NC * 4);
    up(r->st.car_ratio, cr.data(), NC * 8);
    up(r->st.car_speed, cs.data(), NC * 8);
  }
  if (up.e != cudaSuccess) {
    cudaFree(r->buf);
    delete r;
    return cuda_fail("cudaMemcpy(rollouts init)", up.e);
  }
  bool ok = true;
  for (int g = 0; g < pp_rollouts::kGroups; g++) {
    if (cudaStreamCreateWithFlags(&r->gs[g], cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&r->g_done[g], cudaEventDisableTiming) != cudaSuccess)
      ok = false;
  }
  if (cudaEventCreateWithFlags(&r->fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&r->o_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&r->o_join, cudaEventDisableTiming) != cudaSuccess ||
      cudaStreamCreateWithFlags(&r->origin, cudaStreamNonBlocking) != cudaSuccess)
    ok = false;
  if (!ok) {
    cudaError_t e2 = cudaGetLastError();
    pp_rollouts_destroy(r);
    return cuda_fail("rollout streams", e2);
  }
  *out = r;
  return PP_OK;
}

extern "C" void pp_rollouts_destroy(pp_rollouts *r) {
  if (!r) return;
  for (int g = 0; g < pp_rollouts::kGroups; g++) {
    if (r->scratch[g]) cudaFree(r->scratch[g]);
    if (r->gs[g]) cudaStreamDestroy(r->gs[g]);
    if (r->g_done[g]) cudaEventDestroy(r->g_done[g]);
  }
  if (r->fork) cudaEventDestroy(r->fork);
  if (r->graph) cudaGraphExecDestroy(r->graph);
  if (r->origin) cudaStreamDestroy(r->origin);
  if (r->o_fork) cudaEventDestroy(r->o_fork);
  if (r->o_join) cudaEventDestroy(r->o_join);
  if (r->buf) cudaFree(r->buf);
  if (r->tf_buf) cudaFree(r->tf_buf);
  if (r->rc_buf) cudaFree(r->rc_buf);
  if (r->sg_buf) cudaFree(r->sg_buf);
  if (r->rt_buf) cudaFree(r->rt_buf);
  delete r;
}

namespace {

// The k_sim_advance instantiation for (traffic model, recorder on, near-miss measures on).
template <int kTraffic>
auto advance_kernel(bool rec, bool ssm) {
  return rec ? (ssm ? k_sim_advance<kTraffic, true, true> : k_sim_advance<kTraffic, true, false>)
             : (ssm ? k_sim_advance<kTraffic, false, true> : k_sim_advance<kTraffic, false, false>);
}

// dynamic shared memory of the IDM k_sim_advance: S and v (double) and lane (int) per car slot
size_t traffic_smem_bytes(int c) { return (size_t)c * kR * (8 + 8 + 4); }

// One tick of every group: issued on the group streams, forked from / joined to `st`.
// One tick of every group.  Groups are independent (a rollout's tick t+1 depends on its own tick
// t only), so a run forks the group streams off `st` once (`fork`) and joins them once (`join`);
// a captured tick needs both so that the graph is closed.
int issue_tick(pp_rollouts *r, const pp_config *cfg, int32_t consume_k, cudaStream_t st,
               bool fork = true, bool join = true) {
  // device rows of the padded table: logical row 0 starts PPD_PAD_ROWS rows in
  const Track trk{r->map->dev_table + (size_t)PPD_PAD_ROWS * PP_MAP_STRIDE, r->map->n, PP_MAP_STRIDE};
  // groups: contiguous ranges of rollouts, at least 16,384 each, at most 8.  A tick of one group
  // is a chain of eight dependent kernels whose durations simply add up (253 us at 65,536
  // rollouts under ncu, 254 us per tick measured, profiles/r2_rollouts_chain.csv); with several
  // groups different kernels of different groups overlap.  65,536 rollouts, four runs each
  // (profiles/r2_rollouts_groups2.log): 1 group 253-256 M ego-frames/s, 2 groups 271-272 M,
  // 4 groups 270-283 M, 8 groups 254-263 M (64 launches per tick; the host falls behind); any
  // of them loses a run now and then to the shared host (79-183 M).
  // pp_rollouts_set_groups / PP_ROLLOUT_GROUPS override the count (at least 4,096 each then).
  static const int forced_groups = [] {
    const char *e = getenv("PP_ROLLOUT_GROUPS");
    const int v = e && *e ? atoi(e) : 0;
    return v < 0 ? 0 : (v > pp_rollouts::kGroups ? pp_rollouts::kGroups : v);
  }();
  const int forced = r->groups_wanted ? r->groups_wanted : forced_groups;
  int groups = forced ? forced : pp_rollouts::kGroups;
  while (groups > 1 && r->n / groups < (forced ? 4096 : 16384)) groups--;
  const int64_t per = (r->n + groups - 1) / groups;
  const int mc = r->fr.max_cars;
  if (fork) {
    cudaEventRecord(r->fork, st);
    for (int g = 0; g < groups; g++) cudaStreamWaitEvent(r->gs[g], r->fork, 0);
  }
  const int64_t launches0 = pp_launch_count();
  for (int g = 0; g < groups; g++) {
    const int64_t lo = g * per;
    const int64_t cnt = (r->n - lo) < per ? (r->n - lo) : per;
    if (cnt <= 0) continue;
    cudaStream_t gs = r->gs[g];
    const int grid = (int)((cnt + kR - 1) / kR);
    const pp_frames fr = ppi::offset_frames(r->fr, lo);
    const pp_plans pl = ppi::offset_plans(r->pl, lo, mc);
    const bool rec = r->rc.W != 0;
    if (rec)
      k_sim_frames<true><<<grid, kB, 0, gs>>>(trk, lo, cnt, r->c, r->st, r->pl, r->fr, r->rc);
    else
      k_sim_frames<false><<<grid, kB, 0, gs>>>(trk, lo, cnt, r->c, r->st, r->pl, r->fr, r->rc);
    if (!r->scratch[g]) {
      const size_t need = ppi::plan_scratch_bytes(per, mc);
      if (need && cudaMalloc((void **)&r->scratch[g], need) != cudaSuccess)
        return cuda_fail("cudaMalloc(rollout scratch)", cudaGetLastError());
    }
    const bool plan_sums = ppi::plan_adds_checksum(cnt);
    int rc = ppi::plan_batch_scratch(r->map, cfg, &fr, &pl, cnt, gs, r->scratch[g], nullptr,
                                     (unsigned long long *)r->stats_sum + PP_STAT_XSUM);
    if (rc != PP_OK) return rc;
    const bool idm = r->traffic == PP_TRAFFIC_IDM;
    const bool ssm = r->sg_buf != nullptr;
    auto *advance = idm ? advance_kernel<PP_TRAFFIC_IDM>(rec, ssm)
                        : advance_kernel<PP_TRAFFIC_CONSTANT>(rec, ssm);
    advance<<<grid, kB, idm ? traffic_smem_bytes(r->c) : 0, gs>>>(
        trk, lo, cnt, r->c, r->seed, r->first, consume_k, r->st, r->pl,
        (unsigned long long *)r->stats_sum, plan_sums ? 0 : 1, r->mo, r->tf, r->rc, r->sg);
    ppi::count_launch(2);
    if (r->rt_buf) {
      auto *restart = idm ? k_restart<PP_TRAFFIC_IDM> : k_restart<PP_TRAFFIC_CONSTANT>;
      restart<<<(int)((cnt + kB - 1) / kB), kB, 0, gs>>>(trk, lo, cnt, r->c, r->seed, r->first,
                                                          r->st, r->mo, r->tf, r->rt);
      ppi::count_launch(1);
    }
  }
  r->launches_per_tick = pp_launch_count() - launches0;
  if (join) {
    for (int g = 0; g < groups; g++) {
      cudaEventRecord(r->g_done[g], r->gs[g]);
      cudaStreamWaitEvent(st, r->g_done[g], 0);
    }
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail("rollout tick", e);
  return PP_OK;
}

void issue_join_only(pp_rollouts *r, cudaStream_t st) {
  for (int g = 0; g < pp_rollouts::kGroups; g++) {
    cudaEventRecord(r->g_done[g], r->gs[g]);
    cudaStreamWaitEvent(st, r->g_done[g], 0);
  }
}

bool same_cfg(const pp_config &a, const pp_config &b) { return std::memcmp(&a, &b, sizeof a) == 0; }

}  // namespace

extern "C" int pp_rollouts_run(pp_rollouts *r, const pp_config *cfg, int64_t n_ticks,
                               int32_t consume_k, void *cuda_stream) {
  if (!r || !cfg || n_ticks < 0 || consume_k < 1 || consume_k > PP_PATH_LEN - PP_PREV_KEEP)
    return PP_E_ARG;
  cudaStream_t st = (cudaStream_t)cuda_stream;
  if (n_ticks == 0) return PP_OK;
  {
    const int rc = ppi::check_map_device(r->map, "pp_rollouts_run");
    if (rc != PP_OK) return rc;
  }
  if (r->rc.W && (r->rec_k.empty() || r->rec_k.back().second != consume_k))
    r->rec_k.emplace_back(r->tick, consume_k);
  // A tick is ~36 short launches over 8 streams (4 groups, each with its side stream).  It can
  // be captured once and replayed as a CUDA graph (PP_ROLLOUT_GRAPH=1; the pipeline's scratch is
  // owned by the rollouts object, so the graph holds only kernels, memsets and event edges).
  // With enough hardware work queues (pp_api.cu) both ways run at the same, stable speed
  // (≈ 200 M ego-frames/s for 65,536 rollouts on one B200); direct issue is the default because
  // it needs no per-tick join of the groups.
  const bool use_graph = n_ticks >= 8 && getenv("PP_ROLLOUT_GRAPH") != nullptr;
  if (use_graph) {
    cudaStream_t caller = st;
    cudaEventRecord(r->o_fork, caller);
    st = r->origin;
    cudaStreamWaitEvent(st, r->o_fork, 0);
    if (r->graph && (r->graph_k != consume_k || !same_cfg(r->graph_cfg, *cfg))) {
      cudaGraphExecDestroy(r->graph);
      r->graph = nullptr;
    }
    if (!r->graph) {
      // one direct tick first: sizes the stream-ordered pool and sets kernel attributes
      int rc = issue_tick(r, cfg, consume_k, st);
      if (rc != PP_OK) return rc;
      r->tick++;
      n_ticks--;
      cudaGraph_t g = nullptr;
      cudaError_t e = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal);
      if (e != cudaSuccess) return cuda_fail("cudaStreamBeginCapture", e);
      rc = issue_tick(r, cfg, consume_k, st);
      e = cudaStreamEndCapture(st, &g);
      if (rc != PP_OK || e != cudaSuccess) {
        if (g) cudaGraphDestroy(g);
        return rc != PP_OK ? rc : cuda_fail("cudaStreamEndCapture", e);
      }
      e = cudaGraphInstantiate(&r->graph, g, 0);
      cudaGraphDestroy(g);
      if (e != cudaSuccess) {
        r->graph = nullptr;
        return cuda_fail("cudaGraphInstantiate", e);
      }
      r->graph_k = consume_k;
      r->graph_cfg = *cfg;
    }
    for (int64_t t = 0; t < n_ticks; t++) {
      cudaError_t e = cudaGraphLaunch(r->graph, st);
      if (e != cudaSuccess) return cuda_fail("cudaGraphLaunch", e);
      ppi::count_launch((int)r->launches_per_tick);
      r->tick++;
    }
    cudaEventRecord(r->o_join, st);
    cudaStreamWaitEvent(caller, r->o_join, 0);
    return PP_OK;
  }
  for (int64_t t = 0; t < n_ticks; t++) {
    const int rc = issue_tick(r, cfg, consume_k, st, t == 0, t == n_ticks - 1);
    if (rc != PP_OK) {
      issue_join_only(r, st);  // keep `st` ordered after whatever the group streams were given
      return rc;
    }
    r->tick++;
  }
  return PP_OK;
}

extern "C" int pp_rollouts_set_lean(pp_rollouts *r, int lean) {
  if (!r) return PP_E_ARG;
  if (lean && !r->lean) {
    r->full_pl = r->pl;
    pp_plans &p = r->pl;
    p.ego_s = p.ego_d = p.ego_vs = p.ego_vd = p.ego_speed = p.ego_acc = nullptr;
    p.target_speed = p.target_time = nullptr;
    p.next_car_id = p.next_car_in_target_lane = nullptr;
    p.car_d = p.car_vs = p.car_vd = nullptr;
    p.car_next_wp = nullptr;
  } else if (!lean && r->lean) {
    r->pl = r->full_pl;
  }
  r->lean = lean != 0;
  if (r->graph) {  // the captured tick holds the old pointers
    cudaGraphExecDestroy(r->graph);
    r->graph = nullptr;
  }
  return PP_OK;
}

extern "C" int pp_rollouts_set_groups(pp_rollouts *r, int groups) {
  if (!r || groups < 0 || groups > pp_rollouts::kGroups) return PP_E_ARG;
  if (r->graph && groups != r->groups_wanted) {  // the captured tick holds the old split
    cudaGraphExecDestroy(r->graph);
    r->graph = nullptr;
  }
  r->groups_wanted = groups;
  return PP_OK;
}

extern "C" int pp_rollouts_last(const pp_rollouts *r, pp_frames *frames_dev, pp_plans *plans_dev) {
  if (!r) return PP_E_ARG;
  if (frames_dev) *frames_dev = r->fr;
  if (plans_dev) *plans_dev = r->pl;
  return PP_OK;
}

extern "C" int pp_rollouts_get_state(const pp_rollouts *r, pp_rollout_state *h) {
  if (!r || !h) return PP_E_ARG;
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return cuda_fail("pp_rollouts_get_state", e);
  const size_t N = (size_t)r->n, NC = (size_t)r->n * (size_t)r->c;
  const SimState &s = r->st;
  Copy dn{cudaMemcpyDeviceToHost};
  dn(h->ego_x, s.ego_x, N * 8);
  dn(h->ego_y, s.ego_y, N * 8);
  dn(h->ego_yaw_deg, s.ego_yaw, N * 8);
  dn(h->ego_speed_mph, s.ego_mph, N * 8);
  dn(h->path_n, s.path_n, N * 4);
  if (h->path_x || h->path_y) {  // the unconsumed points live in the plan buffer at path_off
    std::vector<int32_t> pn(N), po(N);
    std::vector<double> buf(N * PP_PATH_LEN);
    dn(pn.data(), s.path_n, N * 4);
    dn(po.data(), s.path_off, N * 4);
    for (int axis = 0; axis < 2; axis++) {
      double *dst = axis ? h->path_y : h->path_x;
      if (!dst) continue;
      dn(buf.data(), axis ? r->pl.next_y : r->pl.next_x, N * PP_PATH_LEN * 8);
      for (size_t i = 0; i < N; i++)
        for (int k = 0; k < PP_PATH_LEN; k++)
          dst[i * PP_PATH_LEN + k] = k < pn[i] ? buf[i * PP_PATH_LEN + po[i] + k] : 0.0;
    }
  }
  dn(h->target_lane, s.target_lane, N * 4);
  dn(h->car_lane, s.car_lane, NC * 4);
  dn(h->car_wp, s.car_wp, NC * 4);
  dn(h->car_ratio, s.car_ratio, NC * 8);
  dn(h->car_speed, s.car_speed, NC * 8);
  h->tick = r->tick;
  if (dn.e != cudaSuccess) return cuda_fail("pp_rollouts_get_state copy", dn.e);
  return PP_OK;
}

extern "C" int pp_rollouts_stats(const pp_rollouts *r, int64_t *stats_dev, void *cuda_stream) {
  if (!r || !stats_dev) return PP_E_ARG;
  cudaError_t e = cudaMemcpyAsync(stats_dev, r->stats_sum, PP_STATS_LEN * sizeof(int64_t),
                                  cudaMemcpyDeviceToDevice, (cudaStream_t)cuda_stream);
  if (e != cudaSuccess) return cuda_fail("pp_rollouts_stats", e);
  return PP_OK;
}

extern "C" int pp_rollouts_set_traffic(pp_rollouts *r, int model) {
  if (!r || r->tick != 0 || (model != PP_TRAFFIC_CONSTANT && model != PP_TRAFFIC_IDM))
    return PP_E_ARG;
  r->traffic = model;
  if (model != PP_TRAFFIC_IDM) return PP_OK;
  {
    const int rc = ppi::check_map_device(r->map, "pp_rollouts_set_traffic");
    if (rc != PP_OK) return rc;
  }
  const int nw = r->map->n;
  const size_t N = (size_t)r->n, NC = (size_t)r->n * (size_t)r->c;
  Traffic &tf = r->tf;
  if (!r->tf_buf) {
    cudaError_t e = observer_alloc(r->tf_buf, [&](char *base) {
      ppi::Carve cv(base);
      cv.take(tf.v0, NC);
      cv.take(tf.acc, NC);
      cv.take(tf.cum, 3 * (size_t)(nw + 1));
      cv.take(tf.ego_lanes, 2 * N);
      cv.take(tf.ego_s, 6 * N);
      return cv.size;
    });
    if (e != cudaSuccess) {
      r->traffic = PP_TRAFFIC_CONSTANT;
      return cuda_fail("cudaMalloc(rollout traffic)", e);
    }
  }
  // cum(L, w), summed on the host in ascending w
  std::vector<double> cum(3 * (size_t)(nw + 1));
  for (int L = 0; L < 3; L++) {
    double acc = 0.0;
    cum[(size_t)L * (nw + 1)] = 0.0;
    for (int w = 0; w < nw; w++) {
      acc += r->map->table[(size_t)w * PP_MAP_STRIDE + 10 + L];
      cum[(size_t)L * (nw + 1) + w + 1] = acc;
    }
  }
  cudaError_t e = cudaMemcpy((double *)tf.cum, cum.data(), cum.size() * 8, cudaMemcpyHostToDevice);
  if (e == cudaSuccess && NC) e = cudaMemcpy(tf.v0, r->st.car_speed, NC * 8, cudaMemcpyDeviceToDevice);
  if (e == cudaSuccess && NC) e = cudaMemset(tf.acc, 0, NC * 8);
  if (e != cudaSuccess) {
    r->traffic = PP_TRAFFIC_CONSTANT;
    return cuda_fail("pp_rollouts_set_traffic", e);
  }
  const Track trk{r->map->dev_table + (size_t)PPD_PAD_ROWS * PP_MAP_STRIDE, nw, PP_MAP_STRIDE};
  k_traffic_init<<<(int)((r->n + kB - 1) / kB), kB>>>(trk, r->st.ego_x, r->st.ego_y, tf);
  ppi::count_launch(1);
  e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) {
    r->traffic = PP_TRAFFIC_CONSTANT;
    return cuda_fail("k_traffic_init", e);
  }
  return PP_OK;
}

extern "C" int pp_rollouts_get_traffic(const pp_rollouts *r, pp_rollout_traffic *h) {
  if (!r || !h || r->traffic != PP_TRAFFIC_IDM) return PP_E_ARG;
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return cuda_fail("pp_rollouts_get_traffic", e);
  const size_t N = (size_t)r->n, NC = (size_t)r->n * (size_t)r->c;
  const int buf = (int)(r->tick & 1);  // the copy the next tick reads
  Copy dn{cudaMemcpyDeviceToHost};
  dn(h->car_v0, r->tf.v0, NC * 8);
  dn(h->car_acc, r->tf.acc, NC * 8);
  dn(h->ego_lanes, r->tf.ego_lanes + buf * N, N * 4);
  dn.transpose(h->ego_s, r->tf.ego_s + buf * 3 * N, N, 3);
  if (dn.e != cudaSuccess) return cuda_fail("pp_rollouts_get_traffic copy", dn.e);
  return PP_OK;
}

extern "C" int pp_rollouts_get_incidents(const pp_rollouts *r, pp_rollout_incidents *h) {
  if (!r || !h) return PP_E_ARG;
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return cuda_fail("pp_rollouts_get_incidents", e);
  const size_t N = (size_t)r->n;
  const Monitor &mo = r->mo;
  Copy dn{cudaMemcpyDeviceToHost};
  dn.transpose(h->count, mo.count, N, PP_INC_KINDS);
  dn(h->first_tick, mo.first_tick, N * 8);
  dn(h->first_kind, mo.first_kind, N * 4);
  dn(h->distance_m, mo.dist, N * 8);
  dn(h->clean_m, mo.clean, N * 8);
  dn(h->best_clean_m, mo.best, N * 8);
  dn(h->max_speed, mo.vmax, N * 8);
  dn(h->max_acc, mo.amax, N * 8);
  dn(h->max_jerk, mo.jmax, N * 8);
  if (dn.e != cudaSuccess) return cuda_fail("pp_rollouts_get_incidents copy", dn.e);
  return PP_OK;
}

extern "C" int pp_rollouts_incident_totals(const pp_rollouts *r, int64_t *totals_dev,
                                           void *cuda_stream) {
  if (!r || !totals_dev) return PP_E_ARG;
  return record_totals(r, "pp_rollouts_incident_totals", k_incident_totals, "k_incident_totals",
                       r->mo, PP_INC_TOTALS_LEN, totals_dev, cuda_stream);
}

extern "C" int pp_rollouts_set_recorder(pp_rollouts *r, int32_t window, uint32_t triggers) {
  if (!r || r->tick != 0 || window < 0 || window > PP_REC_MAX_WINDOW ||
      (triggers >> (PP_REC_NONFINITE + 1)) != 0)
    return PP_E_ARG;
  const size_t N = (size_t)r->n;
  Recorder &rc = r->rc;
  auto layout = [&](char *base) {
    ppi::Carve cv(base);
    cv.take(rc.ring, (size_t)window * (size_t)rc.slot_words());
    cv.take(rc.trig_tick, N);
    cv.take(rc.trig_bits, N);
    return cv.size;
  };
  observer_free(r->rc_buf, layout);
  rc.W = 0;
  rc.mask = 0;
  r->rec_k.clear();
  if (window == 0) return PP_OK;
  cudaError_t e = observer_alloc(r->rc_buf, layout);
  if (e != cudaSuccess) return cuda_fail("cudaMalloc(rollout recorder)", e);
  e = cudaMemset(rc.trig_tick, 0xff, N * 8);  // -1: recording
  if (e == cudaSuccess) e = cudaMemset(rc.trig_bits, 0, N * 4);
  if (e != cudaSuccess) {
    observer_free(r->rc_buf, layout);
    return cuda_fail("pp_rollouts_set_recorder", e);
  }
  rc.W = window;
  rc.mask = triggers;
  return PP_OK;
}

extern "C" int pp_rollouts_get_recording(const pp_rollouts *r, const int64_t *rollouts, int64_t m,
                                         pp_rollout_recording *h) {
  if (!r || !h || !r->rc.W || m < 0 || (!rollouts && m != r->n)) return PP_E_ARG;
  for (int64_t i = 0; rollouts && i < m; i++)
    if (rollouts[i] < 0 || rollouts[i] >= r->n) return PP_E_ARG;
  if (m == 0) return PP_OK;
  {
    const int rc = ppi::check_map_device(r->map, "pp_rollouts_get_recording");
    if (rc != PP_OK) return rc;
  }
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return cuda_fail("pp_rollouts_get_recording", e);
  const int W = r->rc.W, c = r->c;
  const size_t M = (size_t)m, MW = M * (size_t)W, MWC = MW * (size_t)c;
  double *const dst_d[10] = {h->ego_x, h->ego_y, h->ego_yaw_deg, h->ego_speed_mph, h->prev_x,
                             h->prev_y, h->car_x, h->car_y, h->car_vx, h->car_vy};
  int32_t *const dst_i[2] = {h->prev_n, h->target_lane_in};
  const size_t words_d[10] = {MW, MW, MW, MW, MW * PP_PREV_KEEP, MW * PP_PREV_KEEP, MWC, MWC, MWC, MWC};
  bool frames = dst_i[0] || dst_i[1];
  for (int f = 0; f < 10; f++) frames = frames || dst_d[f];
  // staging: the rows, the trigger arrays, then (frames only) every frame field
  RecOut out = {};
  int64_t *rows_dev = nullptr;
  auto layout = [&](char *base) {
    ppi::Carve cv(base);
    if (rollouts) cv.take(rows_dev, M);
    cv.take(out.trig_tick, M);
    cv.take(out.trig_bits, M);
    for (int f = 0; frames && f < 10; f++) cv.take(out.d[f], words_d[f]);
    for (int f = 0; frames && f < 2; f++) cv.take(out.i[f], MW);
    return cv.size;
  };
  char *buf = nullptr;
  e = cudaMalloc((void **)&buf, layout(nullptr));
  if (e != cudaSuccess) return cuda_fail("cudaMalloc(recording staging)", e);
  layout(buf);
  if (rollouts) e = cudaMemcpy(rows_dev, rollouts, M * 8, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    const size_t most = frames ? (MWC > MW * PP_PREV_KEEP ? MWC : MW * PP_PREV_KEEP) : M;
    const size_t blocks = (most + kB - 1) / kB;
    const dim3 grid((unsigned)(blocks < 4096 ? (blocks ? blocks : 1) : 4096), frames ? 13 : 1);
    k_rec_gather<<<grid, kB>>>(r->rc, rows_dev, m, r->tick, out);
    ppi::count_launch(1);
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
  }
  std::vector<int64_t> tt(M);
  Copy dn{cudaMemcpyDeviceToHost, e};
  dn(tt.data(), out.trig_tick, M * 8);
  dn(h->trigger_bits, out.trig_bits, M * 4);
  for (int f = 0; frames && f < 10; f++) dn(dst_d[f], out.d[f], words_d[f] * 8);
  for (int f = 0; frames && f < 2; f++) dn(dst_i[f], out.i[f], MW * 4);
  cudaFree(buf);
  if (dn.e != cudaSuccess) return cuda_fail("pp_rollouts_get_recording copy", dn.e);
  // what the host knows: each slot's tick and consume_k, and the constant frame fields
  if (h->trigger_tick) std::memcpy(h->trigger_tick, tt.data(), M * 8);
  for (size_t i = 0; i < M; i++) {
    const int64_t end = tt[i] >= 0 ? tt[i] : r->tick - 1;
    const int64_t filled = end + 1 < W ? end + 1 : W;
    for (int j = 0; j < W; j++) {
      const size_t fi = i * W + j;
      const int64_t t = j < filled ? end - filled + 1 + j : -1;
      if (h->tick) h->tick[fi] = t;
      if (h->consume_k) {
        int32_t k = 0;
        for (const auto &run : r->rec_k)  // a handful of entries: one per change of consume_k
          if (t >= 0 && run.first <= t) k = run.second;
        h->consume_k[fi] = k;
      }
      if (h->n_cars) h->n_cars[fi] = t >= 0 ? c : 0;
      for (int q = 0; h->car_id && q < c; q++) h->car_id[fi * c + q] = t >= 0 ? q : 0;
    }
  }
  return PP_OK;
}

extern "C" int pp_rollouts_set_surrogate(pp_rollouts *r, int on) {
  if (!r || r->tick != 0) return PP_E_ARG;
  const size_t N = (size_t)r->n, M = PP_SSM_MEASURES;
  Surrogate &sg = r->sg;
  auto layout = [&](char *base) {
    ppi::Carve cv(base);
    cv.take(sg.min, M * N);
    cv.take(sg.min_tick, N);
    cv.take(sg.hist, M * PP_SSM_BINS * N);
    return cv.size;
  };
  observer_free(r->sg_buf, layout);
  if (!on) return PP_OK;
  cudaError_t e = observer_alloc(r->sg_buf, layout);
  if (e != cudaSuccess) return cuda_fail("cudaMalloc(rollout surrogate)", e);
  const std::vector<double> inf(M * N, INFINITY);
  e = cudaMemcpy(sg.min, inf.data(), M * N * 8, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemset(sg.min_tick, 0xff, N * 8);  // -1: never lowered
  if (e == cudaSuccess) e = cudaMemset(sg.hist, 0, M * PP_SSM_BINS * N * 4);
  if (e != cudaSuccess) {
    observer_free(r->sg_buf, layout);
    return cuda_fail("pp_rollouts_set_surrogate", e);
  }
  return PP_OK;
}

extern "C" int pp_rollouts_get_surrogate(const pp_rollouts *r, pp_rollout_surrogate *h) {
  if (!r || !h || !r->sg_buf) return PP_E_ARG;
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return cuda_fail("pp_rollouts_get_surrogate", e);
  const size_t N = (size_t)r->n;
  Copy dn{cudaMemcpyDeviceToHost};
  double *const mins[PP_SSM_MEASURES] = {h->min_ttc_front, h->min_ttc_rear, h->min_thw};
  for (int m = 0; m < PP_SSM_MEASURES; m++) dn(mins[m], r->sg.min + m * N, N * 8);
  dn(h->min_ttc_front_tick, r->sg.min_tick, N * 8);
  dn.transpose(h->time_hist, r->sg.hist, N, PP_SSM_MEASURES * PP_SSM_BINS);
  if (dn.e != cudaSuccess) return cuda_fail("pp_rollouts_get_surrogate copy", dn.e);
  return PP_OK;
}

extern "C" int pp_rollouts_surrogate_totals(const pp_rollouts *r, int64_t *totals_dev,
                                            void *cuda_stream) {
  if (!r || !totals_dev || !r->sg_buf) return PP_E_ARG;
  return record_totals(r, "pp_rollouts_surrogate_totals", k_surrogate_totals, "k_surrogate_totals",
                       r->sg, PP_SSM_TOTALS_LEN, totals_dev, cuda_stream);
}

extern "C" int pp_rollouts_set_restart(pp_rollouts *r, uint32_t triggers) {
  if (!r || r->tick != 0 || (triggers >> (PP_REC_NONFINITE + 1)) != 0) return PP_E_ARG;
  const size_t N = (size_t)r->n, K = PP_INC_KINDS, nw = (size_t)r->map->n;
  Restart &rt = r->rt;
  auto layout = [&](char *base) {
    ppi::Carve cv(base);
    cv.take(rt.count0, K * N);
    cv.take(rt.dist0, N);
    cv.take(rt.episodes, N);
    cv.take(rt.by_bit, (K + 1) * N);
    cv.take(rt.ep_tick, N);
    cv.take(rt.ep_m, N);
    cv.take(rt.ended_m, N);
    cv.take(rt.ended_lap, N);
    cv.take(rt.yaw, 3 * nw);
    return cv.size;
  };
  observer_free(r->rt_buf, layout);
  rt.mask = 0;
  if (triggers == 0) return PP_OK;
  {
    const int rc = ppi::check_map_device(r->map, "pp_rollouts_set_restart");
    if (rc != PP_OK) return rc;
  }
  const size_t bytes = layout(nullptr);
  cudaError_t e = observer_alloc(r->rt_buf, layout);
  if (e != cudaSuccess) return cuda_fail("cudaMalloc(rollout restarts)", e);
  // the yaw of a cold start at the centre of lane L on segment w, with create's expression
  const Track trk{r->map->table.data(), r->map->n, PP_MAP_STRIDE};
  std::vector<double> yaw(3 * nw);
  for (int L = 0; L < 3; L++)
    for (int w = 0; w < r->map->n; w++) {
      double x, y, vx, vy;
      trk.car(L, w, 0.0, 1.0, x, y, vx, vy);
      yaw[L * nw + w] = ego_yaw_deg(vx, vy);
    }
  e = cudaMemset(r->rt_buf, 0, bytes);
  if (e == cudaSuccess) e = cudaMemcpy((double *)rt.yaw, yaw.data(), yaw.size() * 8, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    observer_free(r->rt_buf, layout);
    return cuda_fail("pp_rollouts_set_restart", e);
  }
  rt.mask = triggers;
  return PP_OK;
}

extern "C" int pp_rollouts_get_restarts(const pp_rollouts *r, pp_rollout_restarts *h) {
  if (!r || !h || !r->rt_buf) return PP_E_ARG;
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return cuda_fail("pp_rollouts_get_restarts", e);
  const size_t N = (size_t)r->n;
  const Restart &rt = r->rt;
  Copy dn{cudaMemcpyDeviceToHost};
  dn(h->episodes, rt.episodes, N * 8);
  dn.transpose(h->by_bit, rt.by_bit, N, PP_INC_KINDS + 1);
  dn(h->episode_tick, rt.ep_tick, N * 8);
  dn(h->episode_m, rt.ep_m, N * 8);
  dn(h->ended_m, rt.ended_m, N * 8);
  dn(h->ended_lap, rt.ended_lap, N * 8);
  if (dn.e != cudaSuccess) return cuda_fail("pp_rollouts_get_restarts copy", dn.e);
  return PP_OK;
}

extern "C" int pp_rollouts_restart_totals(const pp_rollouts *r, int64_t *totals_dev,
                                          void *cuda_stream) {
  if (!r || !totals_dev || !r->rt_buf) return PP_E_ARG;
  return record_totals(r, "pp_rollouts_restart_totals", k_restart_totals, "k_restart_totals",
                       r->rt, PP_RST_TOTALS_LEN, totals_dev, cuda_stream);
}
