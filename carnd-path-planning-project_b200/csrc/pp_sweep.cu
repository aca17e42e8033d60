// pp_sweep.cu — candidate sweep (BASELINE config 4): 384 candidate trajectories per
// frame through SpeedController / TrajectoryBuilder, scored and argmin-selected.
// Specified in include/pp.h (pp_sweep_batch).
//
// The spline of a candidate depends on the frame and the target lane only, not on the
// target speed / time, so the work is cut as
//   pp_plan_batch   per frame          : ego Frenet state and the planner's own target lane
//   k_sweep_setup   per (frame, lane)  : reference segment, control points, spline fit
//   k_sweep_emit    per candidate      : one block = the 128 candidates of a (frame, lane),
//                                        knots shared in shared memory; emission loop into a
//                                        scorer instead of memory
//   k_sweep_select  warp per frame     : argmin, then the winner's points are emitted again
// This phase is compute bound (FP64 issue): ~3 M instructions per frame against 1.5 KB.
#include <cuda_runtime.h>

#include <cstdio>

#include "pp_device.cuh"
#include "pp_internal.h"

namespace {

using namespace ppd;

constexpr int kCandPerLane = PP_SWEEP_SPEEDS * PP_SWEEP_TIMES;  // 128 = one block
constexpr int kHead = 7;                                        // sc.start, -, -, cx, cy, ca, sa
constexpr int kRows = kHead + 5 * PPD_TAILK;

struct SweepScratch {
  double *est;       // [kRows][3N]  spline state per (frame, lane)
  int32_t *np;       // [3N] kept previous points
  int32_t *code;     // [3N] stored knots | partial << 8 ; 0 = fallback / unusable
  double *scores;    // [N][384]
  int64_t n3;
};

// ego pose as the glue derives it (src/main.cpp:1254-1282): position only
PPD_INLINE void ego_pose(const pp_frames &in, int64_t f, double &x, double &y, int &nprev) {
  if (in.prev_n[f] >= PP_PREV_KEEP) {
    x = in.prev_x[f * PP_PREV_KEEP + PP_PREV_KEEP - 1];
    y = in.prev_y[f * PP_PREV_KEEP + PP_PREV_KEEP - 1];
    nprev = PP_PREV_KEEP;
  } else {
    x = in.ego_x[f];
    y = in.ego_y[f];
    nprev = 0;
  }
}

__global__ void __launch_bounds__(128)
k_sweep_setup(const double *__restrict__ map_table, int n_wp, const __grid_constant__ pp_config cfg,
              const __grid_constant__ pp_frames in, const double *__restrict__ ego_d,
              const double *__restrict__ ego_vd, const double *__restrict__ ego_speed,
              const __grid_constant__ SweepScratch sw, int64_t n) {
  extern __shared__ __align__(16) double s_rows[];  // [PPD_SWEEP_ROWS * PPD_TAILK][blockDim.x]
  MapView m;
  m.t = map_table + PPD_PAD * PP_MAP_STRIDE;
  m.n = n_wp;
  m.pad_lo = n_wp < PPD_PAD ? n_wp : PPD_PAD;
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // frame * 3 + lane
  if (q >= 3 * n) return;
  const int64_t f = q / 3;
  const int lane = (int)(q - f * 3);
  double x, y;
  int nprev;
  ego_pose(in, f, x, y, nprev);
  RefState rs;
  init_reference(m, x, y, rs);
  SpeedCtl sc;
  sc_init(sc, cfg, ego_speed[f]);
  double kept_x[PP_PREV_KEEP], kept_y[PP_PREV_KEEP];  // the kept points are not needed here
  uint32_t flags = 0;
  double *e = sw.est + q;
  KnotSweep ks;
  ks.init(s_rows + threadIdx.x, blockDim.x, e, sw.n3, kHead);
  TrajFrame tf;
  traj_setup(m, cfg, rs, in.prev_x + f * PP_PREV_KEEP, in.prev_y + f * PP_PREV_KEEP, nprev, x, y,
             in.ego_yaw_deg[f], lane, ego_d[f], ego_vd[f], sc, kept_x, kept_y, flags, ks, tf);
  e[0 * sw.n3] = sc.start;
  e[3 * sw.n3] = tf.cx;
  e[4 * sw.n3] = tf.cy;
  e[5 * sw.n3] = tf.ca;
  e[6 * sw.n3] = tf.sa;
  sw.np[q] = tf.np;
  if (tf.fallback) {
    sw.code[q] = 0;
    return;
  }
  const int r0 = ks.r0;
  const int cnt = ks.solve(tf.nk);
  sw.code[q] = cnt | (r0 > 0 ? 1 << 8 : 0);
}

// Scores a trajectory from its points alone (include/pp.h): running |V| sum and max |A|.
struct ScoreOut {
  double px, py, vx, vy, vsum, amax;
  int n;
  PPD_INLINE void init() {
    px = py = vx = vy = vsum = amax = 0;
    n = 0;
  }
  PPD_INLINE void put(int, double x, double y) {
    if (n >= 1) {
      const double nvx = (x - px) * 50, nvy = (y - py) * 50;
      vsum += sqrt(nvx * nvx + nvy * nvy);
      if (n >= 2) {
        const double ax = (nvx - vx) * 50, ay = (nvy - vy) * 50;
        amax = smax(amax, sqrt(ax * ax + ay * ay));
      }
      vx = nvx;
      vy = nvy;
    }
    px = x;
    py = y;
    n++;
  }
  PPD_INLINE void flush() {}
  PPD_INLINE double score(const pp_config &cfg, int lane, int target_lane) const {
    if (n < 3) return PP_SWEEP_BAD;
    const double mean = vsum / (n - 1);
    double over = amax - cfg.maximum_acc;
    if (!(over > 0)) over = 0;
    const double s =
        fabs((double)(lane - target_lane)) + (cfg.max_speed - mean) / cfg.max_speed + 0.5 * over;
    return s < PP_SWEEP_BAD ? s : PP_SWEEP_BAD;  // NaN / inf points (e.g. a standstill) are bad
  }
};

// candidate (iv, it) of a controller that starts at `start`
PPD_INLINE SpeedCtl candidate_ctl(const pp_config &cfg, double start, int iv, int it) {
  SpeedCtl sc;
  sc_init(sc, cfg, start);
  const double v = iv * cfg.max_speed / (PP_SWEEP_SPEEDS - 1);
  const double t = 0.5 * (it + 1);
  sc_limit(sc, v, t);
  return sc;
}

struct SharedKnots {  // the block's (frame, lane) knots, one copy
  const double *base;  // [5][PPD_TAILK]
  int count;
  bool part;
  PPD_INLINE int n() const { return count; }
  PPD_INLINE bool partial() const { return part; }
  PPD_INLINE double x(int i) const { return base[0 * PPD_TAILK + i]; }
  PPD_INLINE double y(int i) const { return base[1 * PPD_TAILK + i]; }
  PPD_INLINE double a(int i) const { return base[2 * PPD_TAILK + i]; }
  PPD_INLINE double b(int i) const { return base[3 * PPD_TAILK + i]; }
  PPD_INLINE double c(int i) const { return base[4 * PPD_TAILK + i]; }
};

__global__ void __launch_bounds__(kCandPerLane)
k_sweep_emit(const __grid_constant__ pp_config cfg, const __grid_constant__ pp_frames in,
             const int32_t *__restrict__ target_lane, const __grid_constant__ SweepScratch sw,
             int64_t n) {
  __shared__ double s_knots[5 * PPD_TAILK];
  __shared__ double s_head[kHead];
  const int64_t q = blockIdx.x;  // frame * 3 + lane
  const int64_t f = q / 3;
  const int lane = (int)(q - f * 3);
  const int code = sw.code[q];
  for (int i = threadIdx.x; i < 5 * PPD_TAILK; i += blockDim.x) s_knots[i] = sw.est[(kHead + i) * sw.n3 + q];
  if (threadIdx.x < kHead) s_head[threadIdx.x] = sw.est[threadIdx.x * sw.n3 + q];
  __syncthreads();
  const int iv = threadIdx.x / PP_SWEEP_TIMES, it = threadIdx.x % PP_SWEEP_TIMES;
  double *dst = sw.scores + f * PP_SWEEP_CANDS + (int64_t)lane * kCandPerLane + threadIdx.x;
  if (code == 0) {
    *dst = PP_SWEEP_BAD;
    return;
  }
  const SpeedCtl sc = candidate_ctl(cfg, s_head[0], iv, it);
  ScoreOut so;
  so.init();
  const int np = sw.np[q];
  for (int i = 0; i < np; i++) so.put(i, in.prev_x[f * PP_PREV_KEEP + i], in.prev_y[f * PP_PREV_KEEP + i]);
  SharedKnots kn{s_knots, code & 0xff, (code >> 8) != 0};
  uint32_t flags = 0;
  int bail;
  // the emission kernel's lean loop first; a candidate with an operand it does not cover
  // (bail 5: e.g. a standstill's zero chord) is redone on the complete loop — same values
  traj_emit_lean(kn, cfg, sc, s_head[3], s_head[4], s_head[5], s_head[6], np, so, flags, bail);
  if (bail == 5) {
    so.init();
    for (int i = 0; i < np; i++)
      so.put(i, in.prev_x[f * PP_PREV_KEEP + i], in.prev_y[f * PP_PREV_KEEP + i]);
    flags = 0;
    traj_emit(kn, cfg, sc, s_head[3], s_head[4], s_head[5], s_head[6], np, so, flags, bail);
  }
  // (bail 1 — a spline argument at or left of the first staged knot, which lies LEFT of the
  // local origin — needs the loop to walk backwards, i.e. a negative speed.  A candidate's ramp
  // runs from the ego speed (a norm, >= 0) to v_i >= 0 and acceleration overrides only cap
  // increases, so no candidate gets there; were it to happen it would be scored BAD here.)
  *dst = bail ? PP_SWEEP_BAD : so.score(cfg, lane, target_lane[f]);
}

// warp per frame: argmin (lowest index on ties), then lane 0 emits the winner's points
__global__ void __launch_bounds__(128)
k_sweep_select(const __grid_constant__ pp_config cfg, const __grid_constant__ pp_frames in,
               const __grid_constant__ SweepScratch sw, const __grid_constant__ pp_sweep_out out,
               int64_t n) {
  __shared__ double s_knots[4][5 * PPD_TAILK];
  const int wib = threadIdx.x >> 5, ln = threadIdx.x & 31;
  const int64_t f = (int64_t)blockIdx.x * 4 + wib;
  if (f >= n) return;
  const double *sc_row = sw.scores + f * PP_SWEEP_CANDS;
  double best = 0;
  int arg = -1;
  for (int i = ln; i < PP_SWEEP_CANDS; i += 32) {
    const double v = sc_row[i];
    if (out.scores) out.scores[f * PP_SWEEP_CANDS + i] = v;
    if (arg < 0 || v < best) {  // ascending i within a lane: strict < keeps the lowest index
      best = v;
      arg = i;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ob = __shfl_down_sync(0xffffffffu, best, o);
    const int oa = __shfl_down_sync(0xffffffffu, arg, o);
    if (oa >= 0 && (arg < 0 || ob < best || (ob == best && oa < arg))) {
      best = ob;
      arg = oa;
    }
  }
  arg = __shfl_sync(0xffffffffu, arg, 0);
  best = __shfl_sync(0xffffffffu, best, 0);
  const int lane = arg / kCandPerLane, rest = arg % kCandPerLane;
  const int64_t q = f * 3 + lane;
  for (int i = ln; i < 5 * PPD_TAILK; i += 32) s_knots[wib][i] = sw.est[(kHead + i) * sw.n3 + q];
  __syncwarp();
  if (ln != 0) return;
  out.best[f] = arg;
  out.best_score[f] = best;
  double *ox = out.next_x + f * PP_PATH_LEN, *oy = out.next_y + f * PP_PATH_LEN;
  const int code = sw.code[q];
  int np = 0;
  if (code != 0 && best < PP_SWEEP_BAD) {
    np = sw.np[q];
    for (int i = 0; i < np; i++) {
      ox[i] = in.prev_x[f * PP_PREV_KEEP + i];
      oy[i] = in.prev_y[f * PP_PREV_KEEP + i];
    }
    const SpeedCtl sc = candidate_ctl(cfg, sw.est[0 * sw.n3 + q], rest / PP_SWEEP_TIMES,
                                      rest % PP_SWEEP_TIMES);
    SharedKnots kn{s_knots[wib], code & 0xff, (code >> 8) != 0};
    ArrayOut pts{ox, oy};
    uint32_t flags = 0;
    int bail;
    np = traj_emit(kn, cfg, sc, sw.est[3 * sw.n3 + q], sw.est[4 * sw.n3 + q],
                          sw.est[5 * sw.n3 + q], sw.est[6 * sw.n3 + q], np, pts, flags, bail);
  }
  for (int i = np; i < PP_PATH_LEN; i++) {
    ox[i] = __longlong_as_double(0x7ff8000000000000ll);
    oy[i] = __longlong_as_double(0x7ff8000000000000ll);
  }
  out.n_points[f] = np;
}

}  // namespace

extern "C" int pp_sweep_batch(const pp_map *map, const pp_config *cfg, const pp_frames *in,
                              const pp_sweep_out *out, int64_t n, void *cuda_stream) {
  if (!map || !cfg || !in || !out || n < 0) return PP_E_ARG;
  if (!out->best || !out->best_score || !out->next_x || !out->next_y || !out->n_points)
    return PP_E_ARG;
  {
    const int rc = ppi::check_map_device(map, "pp_sweep_batch");
    if (rc != PP_OK) return rc;
  }
  if (n == 0) return PP_OK;
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const size_t N = (size_t)n;
  // scratch: plans of the ordinary step (for ego_d, ego_vd, ego_speed, target_lane) + sweep state
  pp_plans pl = {};
  SweepScratch sw;
  auto carve = [&](char *base) {
    ppi::Carve cv(base);
    cv.take(pl.next_x, N * PP_PATH_LEN);
    cv.take(pl.next_y, N * PP_PATH_LEN);
    cv.take(pl.n_points, N);
    cv.take(pl.ego_lane, N);
    cv.take(pl.ref_wp, N);
    cv.take(pl.target_lane, N);
    cv.take(pl.flags, N);
    cv.take(pl.ego_d, N);
    cv.take(pl.ego_vd, N);
    cv.take(pl.ego_speed, N);
    cv.take(sw.est, (size_t)kRows * 3 * N);
    cv.take(sw.np, 3 * N);
    cv.take(sw.code, 3 * N);
    cv.take(sw.scores, N * PP_SWEEP_CANDS);
    return cv.size;
  };
  char *buf = nullptr;
  cudaError_t e = cudaMallocAsync((void **)&buf, carve(nullptr), st);
  if (e != cudaSuccess) {
    ppi::set_cuda_error("cudaMallocAsync(sweep)", (int)e, cudaGetErrorString(e));
    cudaGetLastError();
    return PP_E_CUDA;
  }
  carve(buf);
  sw.n3 = 3 * n;
  int rc = pp_plan_batch(map, cfg, in, &pl, n, st);
  if (rc == PP_OK) {
    const size_t smem_setup = (size_t)PPD_SWEEP_ROWS * PPD_TAILK * 128 * sizeof(double);
    static bool attr_done = false;
    if (!attr_done) {
      cudaFuncSetAttribute(k_sweep_setup, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_setup);
      attr_done = true;
    }
    k_sweep_setup<<<(unsigned)((3 * n + 127) / 128), 128, smem_setup, st>>>(
        map->dev_table, map->n, *cfg, *in, pl.ego_d, pl.ego_vd, pl.ego_speed, sw, n);
    k_sweep_emit<<<(unsigned)(3 * n), kCandPerLane, 0, st>>>(*cfg, *in, pl.target_lane, sw, n);
    k_sweep_select<<<(unsigned)((n + 3) / 4), 128, 0, st>>>(*cfg, *in, sw, *out, n);
    ppi::count_launch(3);
    cudaError_t le = cudaGetLastError();
    if (le != cudaSuccess) {
      ppi::set_cuda_error("sweep kernels", (int)le, cudaGetErrorString(le));
      rc = PP_E_CUDA;
    }
  }
  cudaFreeAsync(buf, st);
  return rc;
}
