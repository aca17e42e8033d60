/* pp.h — C ABI of the B200-native batched highway path planner.
 *
 * One call, pp_plan_batch, replaces the planning step that the reference runs
 * once per telemetry message inside main::onMessage
 * (reference src/main.cpp:1254-1457): ego state from the 10th reused point,
 * Map::init_reference_waypoint / lane_matching / project_speed, the
 * sensor-fusion matching loop, LaneChangePlanner::calculate_target_lane,
 * LimitSpeed::calculate, SpeedController and TrajectoryBuilder::build
 * (tk::spline fit + 0.02 s point emission) — for N independent frames at once,
 * on the GPU, over struct-of-arrays frame buffers.
 *
 * The reference has no FFI of its own for this path (the path is inlined in a
 * lambda whose only interface is the simulator wire message), so every entry
 * point below cites the reference lines whose behaviour it reproduces.
 *
 * Conventions
 *   - plain C, no exceptions cross this boundary; every function returns
 *     PP_OK (0) or a negative PP_E_* code; pp_strerror() names it.
 *   - "dev" pointers are CUDA device pointers on the device that was current
 *     when the pp_map was created; "host" pointers are ordinary (ideally
 *     pinned) host memory.  The caller owns every buffer; the library owns
 *     pp_map.  A call made while another device is current fails with
 *     PP_E_ARG (one pp_map per device).
 *   - pp_plan_batch is asynchronous on the caller's stream and re-entrant:
 *     the reference keeps reference_waypoint_id/ratio as mutable state on
 *     the shared Map (src/main.cpp:132-133); here that state lives in
 *     registers per frame, so the map is immutable after creation.
 *   - There is NO CPU planning path in this library.  If the CUDA device or
 *     kernels are unavailable the calls fail with PP_E_CUDA.
 */
#ifndef PP_B200_H
#define PP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PP_VERSION 102

/* Fixed sizes of the reference's planning step. */
#define PP_NUM_LANES 3    /* src/main.cpp:22  NUM_LANES */
#define PP_PREV_KEEP 10   /* src/main.cpp:1258 prev_trajectory_length */
#define PP_PATH_LEN 50    /* src/main.cpp:854,1039 result_points.size() < 50 */
#define PP_MAX_CARS 64    /* largest n_cars per frame this build accepts (BASELINE config 5) */

/* One row of the uploaded map table (doubles per waypoint):
 * ref.x ref.y c0.x c0.y c1.x c1.y c2.x c2.y nx ny len0 len1 len2
 * = Map::Waypoint (src/main.cpp:76-82) plus get_lane_length(i, lane)
 * (src/main.cpp:138-142) precomputed with the same expression. */
#define PP_MAP_STRIDE 13

/* Error codes. */
#define PP_OK 0
#define PP_E_ARG (-1)      /* null pointer / bad size */
#define PP_E_CUDA (-2)     /* CUDA runtime error (pp_last_cuda_error() has the text) */
#define PP_E_IO (-3)       /* map file could not be read */
#define PP_E_NOMEM (-4)
#define PP_E_RANGE (-5)    /* n_cars > PP_MAX_CARS, n_waypoints out of range, ... */

/* Per-frame flag bits: one bit per print / log site of the reference, so
 * that anomalies are data and never abort the batch (SURVEY §5). */
#define PP_F_EGO_MATCH_FAIL   (1u << 0)  /* src/main.cpp:1304 "can't lane match ego" */
#define PP_F_CAR_DROPPED      (1u << 1)  /* :1338 car failed lane_matching, erased */
#define PP_F_COLLISION        (1u << 2)  /* :1077 "detected collision" */
#define PP_F_BRAKE            (1u << 3)  /* :1109 */
#define PP_F_MAXBRAKE         (1u << 4)  /* :1101 */
#define PP_F_ADJUST           (1u << 5)  /* :1131 */
#define PP_F_KEEP             (1u << 6)  /* :1146 */
#define PP_F_SPLINE_INPUT_ERR (1u << 7)  /* :837 non-increasing knot x, truncated */
#define PP_F_FALLBACK         (1u << 8)  /* :848 angle-based generator taken (silent in the reference) */
#define PP_F_ACC_OVERRIDE     (1u << 9)  /* :964 */
#define PP_F_CURV_ADJUST      (1u << 10) /* :988 */
#define PP_F_LANE_SWITCH_NEG  (1u << 11) /* :711 */
#define PP_F_VETO             (1u << 12) /* :1366 "target lane too far" */
#define PP_F_ACCT_HIGH        (1u << 13) /* :950 */
#define PP_F_ACCN_HIGH        (1u << 14) /* :978 */
#define PP_F_SPLINE_WARNING   (1u << 15) /* :927 */
#define PP_F_CLOSED_RANGE     (1u << 16) /* :408 condition true for some car */
#define PP_F_CLOSED_AHEAD     (1u << 17) /* :423 condition true for some car */
#define PP_F_CLOSED_BEHIND    (1u << 18) /* :439 condition true for some car */
#define PP_F_TRANSFORM_ERR    (1u << 19) /* :1015 */
#define PP_F_COLD_START       (1u << 20) /* :1261 fewer than 10 previous points */
#define PP_NUM_FLAGS 21

typedef struct pp_map pp_map; /* opaque: host table + device copy */

/* Tunables = the reference's globals (src/main.cpp:30,39-49).
 * pp_config_default() fills in exactly those literals. */
typedef struct pp_config {
  double relaxed_acc;                   /* 5    :39 */
  double min_relaxed_acc_while_braking; /* 4    :40 */
  double maximum_acc;                   /* 8    :42 */
  double max_speed;                     /* 22.2 :45 */
  double car_length;                    /* 4.5  :46 */
  double safety_distance;               /* 2    :47 */
  double keep_distance;                 /* 10   :48 */
  double keep_distance_leeway;          /* 0.5  :49 */
  int32_t test_fast_lane_change;        /* 0    :30 */
  int32_t reserved;
} pp_config;

/* Input frames, struct of arrays, N frames.  Inner arrays are frame-major:
 * prev_x[f*PP_PREV_KEEP + i], car_x[f*max_cars + j].
 * Fields mirror the telemetry the reference reads (src/main.cpp:1233-1252,
 * 1297,1328-1334); the unused wire fields (s, d, end_path_s/d, car s/d) are
 * not carried.  Car ids within one frame must be distinct (the reference's map keeps the
 * LAST row of a repeated id; pp::wire::parse_telemetry applies that rule); cars may appear
 * in any order (the reference iterates a std::map<int,Car>, i.e. ascending id, and only
 * tie-breaks depend on that order — reproduced here by id). */
typedef struct pp_frames {
  const double *ego_x;         /* [N] telemetry x  (used when prev_n < 10, :1233) */
  const double *ego_y;         /* [N] */
  const double *ego_yaw_deg;   /* [N] degrees; heading fallback only (:587,596,604) */
  const double *ego_speed_mph; /* [N] used when prev_n < 10 (:1238-1239) */
  const int32_t *prev_n;       /* [N] previous_path size; only ">= 10" matters (:1261) */
  const double *prev_x;        /* [N][10] first 10 points of previous_path_x */
  const double *prev_y;        /* [N][10] */
  const int32_t *target_lane_in; /* [N] persistent target_lane (:1195,1355) */
  const int32_t *n_cars;       /* [N] 0..max_cars */
  const int32_t *car_id;       /* [N][max_cars] */
  const double *car_x;         /* [N][max_cars] */
  const double *car_y;
  const double *car_vx;
  const double *car_vy;
  int32_t max_cars;            /* row length of the car arrays, <= PP_MAX_CARS */
  int32_t reserved;
  /* Optional, all five NULL or all five set: cars the reference still holds in its persistent
   * std::map<int,Car> although the current message does not list them (src/main.cpp:1194,
   * 1325-1334 only touch the cars of the message).  Such a car takes part in the planning with
   * the Frenet values of its last sighting, which the reference never recomputes:
   * car_frozen_lane[f*max_cars + j] >= 0 marks slot j as frozen (lane = that value, s / d / vs /
   * vd from the arrays below; its car_x / car_y are not matched, car_vx / car_vy still give its
   * Cartesian speed to LimitSpeed, :1080); -1 = an ordinary car of the current message.
   * include/pp_wire.hpp (pp::wire::Session) maintains this state for replayed sessions. */
  const int32_t *car_frozen_lane; /* [N][max_cars] */
  const double *car_frozen_s;     /* [N][max_cars] */
  const double *car_frozen_d;
  const double *car_frozen_vs;
  const double *car_frozen_vd;
} pp_frames;

/* Output plans, struct of arrays.  next_x/next_y entries at and beyond
 * n_points are set to quiet NaN.  Any pointer in the "diagnostics" and "per-car" groups may
 * be NULL (that output is then skipped). */
typedef struct pp_plans {
  double *next_x;        /* [N][50]  (:1450-1462) */
  double *next_y;        /* [N][50] */
  int32_t *n_points;     /* [N] <= 50 (10 kept + <= 40 new; fewer only in the fallback) */
  int32_t *ego_lane;     /* [N] */
  int32_t *ref_wp;       /* [N] reference_waypoint_id, un-wrapped, 0..n_wp (:186) */
  int32_t *target_lane;  /* [N] after planner + veto: the state carried to the next frame */
  uint32_t *flags;       /* [N] PP_F_* */
  /* diagnostics */
  double *ego_s, *ego_d, *ego_vs, *ego_vd;  /* [N] (:1302,1313) */
  double *ego_speed, *ego_acc;              /* [N] (:1273-1276,1319-1320) */
  double *target_speed, *target_time;       /* [N] SpeedController after both limits (:1430,1437) */
  int32_t *next_car_id;                     /* [N] -1 if none (:1383-1400) */
  int32_t *next_car_in_target_lane;         /* [N] -1 if none (:1402-1411) */
  /* per-car results of the sensor-fusion matching loop (:1325-1350) */
  double *car_s, *car_d, *car_vs, *car_vd;  /* [N][max_cars] */
  int32_t *car_lane;                        /* [N][max_cars]; -1 = dropped */
  int32_t *car_next_wp;                     /* [N][max_cars] un-wrapped */
} pp_plans;

/* Aggregate statistics vector (all int64 so that sums are exact and the
 * 1/2/4/8-GPU all-reduce is bit-identical; SURVEY §8e). */
#define PP_STAT_FRAMES 0
#define PP_STAT_POINTS 1                         /* sum of n_points */
#define PP_STAT_TARGET_LANE0 2                   /* +lane */
#define PP_STAT_EGO_LANE0 5                      /* +lane */
#define PP_STAT_LANE_CHANGES 8                   /* target_lane != ego_lane */
#define PP_STAT_FLAG0 9                          /* +bit, PP_NUM_FLAGS entries */
#define PP_STAT_XSUM (PP_STAT_FLAG0 + PP_NUM_FLAGS) /* fixed-point checksum of emitted x,y */
#define PP_STATS_LEN (PP_STAT_XSUM + 1)

int pp_version(void);
/* Optional, before the process's first CUDA call: asks for 32 hardware work queues
 * (CUDA_DEVICE_MAX_CONNECTIONS, unless the environment already sets it).  The planner keeps up
 * to nine streams busy; with the default 8 queues independent streams share a queue and
 * serialise (DESIGN.md §9.1).  The library never changes the environment by itself. */
int pp_init(void);
const char *pp_strerror(int code);
const char *pp_last_cuda_error(void);
int pp_device_count(void); /* number of CUDA devices, or PP_E_CUDA */

/* Defaults = the literals at src/main.cpp:30,39-49. */
int pp_config_default(pp_config *cfg);

/* Map::Init (src/main.cpp:89-131) on the host (same libm as the reference, so
 * the table is bit-identical), then one upload to the current device. */
int pp_map_create(const double *wx, const double *wy, int n, pp_map **out);
/* CSV loader with the reference's parsing (x,y as double; columns 3-5 ignored;
 * src/main.cpp:1171-1191). */
int pp_map_create_from_csv(const char *path, pp_map **out);
void pp_map_destroy(pp_map *map);
int pp_map_num_waypoints(const pp_map *map);
/* Copy the host table out: n * PP_MAP_STRIDE doubles. */
int pp_map_table(const pp_map *map, double *out);

/* The hot path.  in/out hold DEVICE pointers.  Asynchronous on `cuda_stream`
 * (a cudaStream_t, may be NULL for the default stream). */
int pp_plan_batch(const pp_map *map, const pp_config *cfg, const pp_frames *in,
                  const pp_plans *out, int64_t n_frames, void *cuda_stream);

/* Same call with HOST buffers: uploads the inputs, plans, downloads the
 * outputs (chunked, copies overlapped with compute), returns when the host
 * buffers are complete.  This is the drop-in for a CPU caller. */
int pp_plan_batch_host(const pp_map *map, const pp_config *cfg, const pp_frames *in,
                       const pp_plans *out, int64_t n_frames);

/* The same call for a caller that does not want its own points sent back over PCIe.  A frame
 * with prev_n >= PP_PREV_KEEP keeps its first PP_PREV_KEEP previous points as the first points
 * of the new trajectory, verbatim (result_points = prev_trajectory, src/main.cpp:578,
 * 1446-1452) — the caller already holds them in in->prev_x / in->prev_y.  Here a trajectory
 * comes back in two parts, and out->next_x / out->next_y must be NULL:
 *   tail_x, tail_y [n][PP_PATH_LEN - PP_PREV_KEEP]  points PP_PREV_KEEP.. of every frame;
 *   head_x, head_y [n][PP_PREV_KEEP]                points 0..PP_PREV_KEEP-1.  The library writes
 *       a head row ONLY for a frame that kept nothing (prev_n < PP_PREV_KEEP: all its points are
 *       new); every other row is left as the caller has it.  head_x / head_y may be the very
 *       buffers passed as in->prev_x / in->prev_y (they are read before they are written), and
 *       then hold the first points of every trajectory on return.
 * head ++ tail of frame i equals row i of pp_plan_batch_host's next_x / next_y bit for bit
 * (tests/test_gpu_parity.py); 160 of the 820 bytes per frame stay off the bus. */
typedef struct pp_split_rows {
  double *head_x, *head_y;
  double *tail_x, *tail_y;
} pp_split_rows;
int pp_plan_batch_host_split(const pp_map *map, const pp_config *cfg, const pp_frames *in,
                             const pp_plans *out, const pp_split_rows *rows, int64_t n_frames);

/* Aggregate statistics of a planned batch on the device:
 * stats_dev[PP_STATS_LEN] (int64, overwritten).  The multi-GPU job all-reduces
 * this vector (pp_stats_reduce, ncclSum) — the only collective on the path. */
int pp_stats_batch(const pp_plans *plans_dev, int64_t n_frames, int64_t *stats_dev,
                   void *cuda_stream);

/* f64 minimum / maximum statistics of a planned batch (SURVEY §8e), computed from the plan
 * outputs alone so that any caller can re-derive them: with V_k = (P_{k+1} - P_k) * 50 and
 * A_k = (V_{k+1} - V_k) * 50 over a frame's n_points output points (k < n_points - 1 and
 * k < n_points - 2), every operation in IEEE double, left to right, no fused multiply-add.
 * Non-finite values do not take part; an entry nothing contributed to stays at +inf (minima)
 * or -inf (maxima).  ego_speed / target_speed are optional outputs of pp_plans. */
#define PP_FSTAT_MIN_EGO_SPEED 0     /* min over frames of ego_speed (:1273) */
#define PP_FSTAT_MIN_TARGET_SPEED 1  /* ... of the SpeedController target (:1430,1437) */
#define PP_FSTAT_MIN_STEP_SPEED 2    /* min over frames and k of |V_k| */
#define PP_FSTAT_NMIN 3              /* entries [0, NMIN) reduce with min, the rest with max */
#define PP_FSTAT_MAX_EGO_SPEED 3
#define PP_FSTAT_MAX_TARGET_SPEED 4
#define PP_FSTAT_MAX_STEP_SPEED 5    /* max |V_k| */
#define PP_FSTAT_MAX_ACC 6           /* max |A_k|: peak total acceleration along the plans
                                        (acc_T and acc_N of :930-944 combined) */
#define PP_FSTATS_LEN 7
/* fstats_dev[PP_FSTATS_LEN] (device, double, overwritten); asynchronous on cuda_stream. */
int pp_fstats_batch(const pp_plans *plans_dev, int64_t n_frames, double *fstats_dev,
                    void *cuda_stream);

/* ---- the one collective of a multi-GPU job: the final reduction of the statistics ----
 * Frames are independent, so a job shards them contiguously over the GPUs (rank r plans
 * [r N / G, (r + 1) N / G)) and exchanges nothing until every shard is planned; then
 * pp_stats_reduce all-reduces, in place and as one NCCL group on cuda_stream, the int64 vector
 * (ncclSum — exact, so 1/2/4/8-GPU results are identical) and the f64 vector (ncclMin over
 * [0, PP_FSTAT_NMIN), ncclMax over the rest); either pointer may be NULL.  nccl_comm is an
 * ncclComm_t: the caller's own, or one made by the helpers below (one process per GPU: rank 0
 * calls pp_comm_unique_id and ships the PP_COMM_ID_BYTES to the others by any means, every
 * rank calls pp_comm_init_rank with its device current; one process driving several devices:
 * pp_comm_init_all, and the per-device pp_stats_reduce calls between pp_comm_group_begin / _end).
 * NCCL is loaded at run time (the copy already in the process if there is one). */
#define PP_COMM_ID_BYTES 128
int pp_comm_unique_id(void *id_out);
int pp_comm_init_rank(const void *id, int rank, int world, void **nccl_comm_out);
int pp_comm_init_all(int n_dev, const int *devices, void **nccl_comms_out);
int pp_comm_destroy(void *nccl_comm);
int pp_comm_group_begin(void);
int pp_comm_group_end(void);
int pp_stats_reduce(void *nccl_comm, int64_t *stats_dev, double *fstats_dev, void *cuda_stream);

/* pp_plan_batch followed by pp_stats_batch in one call (stats_dev[PP_STATS_LEN], overwritten):
 * the statistics of each chunk are taken as soon as the chunk is planned, concurrently with
 * the planning of the other chunks.  Same results as the two separate calls. */
int pp_plan_stats_batch(const pp_map *map, const pp_config *cfg, const pp_frames *in,
                        const pp_plans *out, int64_t n_frames, int64_t *stats_dev,
                        void *cuda_stream);

/* Kernel selection for pp_plan_batch: 0 = auto (the pipeline; below 1536 frames the
 * warp-per-frame kernel), 1 = one thread per frame in a single kernel, 2 = the pipeline
 * (k_prep, k_cars, k_decide_t, k_emit), 3 = the pipeline with the tiled cars kernel (a warp's
 * frames' cars by TMA into shared memory, reductions in the same kernel), 4 = one warp per
 * frame (lowest latency: closest-waypoint argmin and the per-car work spread over the lanes).
 * All variants produce the same bits. */
int pp_set_kernel_variant(int variant);
/* Chunks of a large batch that pp_plan_batch keeps in flight at once on internal streams:
 * 1..8, 0 = default (4).  1 runs the kernels of the pipeline strictly one after the other,
 * which is what a per-kernel time breakdown needs. */
int pp_set_pipes(int pipes);
/* Measurement aid (bench.py): when on, pp_plan_batch records CUDA events on the
 * caller's stream around each kernel of the pipeline.  pp_get_phase_ms waits for
 * the last of them and returns the summed device time in ms of ms_out[0] = ego
 * preparation, [1] = per-car matching, [2] = decision + spline fit, [3] = point
 * emission, [4] = complete path for the queued rare frames (PP_NUM_PHASES
 * values) over all chunks launched since the previous call (chunks_out, may be
 * NULL). */
#define PP_NUM_PHASES 5
int pp_set_phase_timing(int on);
int pp_get_phase_ms(double *ms_out, int64_t *chunks_out);
/* Number of kernel launches issued by this library since load (bench.py's
 * gpu_launches). */
int64_t pp_launch_count(void);

/* ---- unit-level entry points (device pointers), one per reference function.
 * Each runs the same __device__ code the fused kernel uses. ---- */

/* distancesq_pt_seg (src/helpers.h:188-249): out_d2, out_rnom, out_rdenom, out_snom [n]. */
int pp_distancesq_pt_seg_batch(const double *px, const double *py, const double *ax,
                               const double *ay, const double *bx, const double *by,
                               double *out_d2, double *out_rnom, double *out_rdenom,
                               double *out_snom, int64_t n, void *cuda_stream);

/* Map::init_reference_waypoint (src/main.cpp:143-197) for n points:
 * out_ref_wp[n], out_ratio[n][3]. */
int pp_init_reference_waypoint_batch(const pp_map *map, const double *x, const double *y,
                                     int32_t *out_ref_wp, double *out_ratio, int64_t n,
                                     void *cuda_stream);

/* Map::lane_matching + project_speed (src/main.cpp:199-275,330-358) for n
 * objects, each relative to its own reference point (rx, ry):
 * out_ok, out_lane, out_next_wp [n] ; out_s, out_d, out_vs, out_vd [n]. */
int pp_lane_matching_batch(const pp_map *map, const double *rx, const double *ry,
                           const double *x, const double *y, const double *vx,
                           const double *vy, int32_t *out_ok, int32_t *out_lane,
                           int32_t *out_next_wp, double *out_s, double *out_d,
                           double *out_vs, double *out_vd, int64_t n, void *cuda_stream);

/* Map::project_speed (src/main.cpp:330-358) alone: speed vectors (vx, vy)[n]
 * against the reference-line segment ending at waypoint next_wp[n] (un-wrapped
 * ids as lane_matching returns them): out_vs, out_vd [n]. */
int pp_project_speed_batch(const pp_map *map, const double *vx, const double *vy,
                           const int32_t *next_wp, double *out_vs, double *out_vd, int64_t n,
                           void *cuda_stream);

/* Map::get_lane_pos (src/main.cpp:277-328) relative to (rx, ry):
 * out_x, out_y, out_dist [n]; out_wp [n]. */
int pp_get_lane_pos_batch(const pp_map *map, const double *rx, const double *ry,
                          const double *s, const int32_t *lane, double *out_x,
                          double *out_y, int32_t *out_wp, double *out_dist, int64_t n,
                          void *cuda_stream);

/* tk::spline::set_points + operator() (src/spline.h:284-396): n_splines
 * splines of n_knots (3..15) knots each, knots[k*n_splines... ] laid out
 * spline-major: kx[i*n_knots + k]; each evaluated at n_q query points
 * q[i*n_q + j] -> out[i*n_q + j]. */
int pp_spline_batch(const double *kx, const double *ky, int32_t n_knots, const double *q,
                    int32_t n_q, double *out, int64_t n_splines, void *cuda_stream);

/* Udacity starter helpers (src/helpers.h:43-155); never called by the
 * reference's planner but part of its API surface. maps_* are device arrays
 * of n_wp entries. */
int pp_closest_waypoint_batch(const double *x, const double *y, const double *maps_x,
                              const double *maps_y, int32_t n_wp, int32_t *out, int64_t n,
                              void *cuda_stream);
int pp_next_waypoint_batch(const double *x, const double *y, const double *theta,
                           const double *maps_x, const double *maps_y, int32_t n_wp,
                           int32_t *out, int64_t n, void *cuda_stream);
int pp_get_frenet_batch(const double *x, const double *y, const double *theta,
                        const double *maps_x, const double *maps_y, int32_t n_wp,
                        double *out_s, double *out_d, int64_t n, void *cuda_stream);
int pp_get_xy_batch(const double *s, const double *d, const double *maps_s,
                    const double *maps_x, const double *maps_y, int32_t n_wp, double *out_x,
                    double *out_y, int64_t n, void *cuda_stream);

/* LaneChangePlanner::calculate_target_lane (src/main.cpp:364-485) on explicit,
 * already matched cars: problem i has n_cars cars car_*[i*n_cars + j] (lane < 0
 * = car not in the map) and scalars ego_lane/target_lane/ego_s/ego_vs/dt0 [n].
 * out_target_lane[n]. */
int pp_lane_change_batch(const pp_config *cfg, const int32_t *car_id, const double *car_s,
                         const double *car_vs, const int32_t *car_lane, int32_t n_cars,
                         const int32_t *ego_lane, const int32_t *target_lane, const double *ego_s,
                         const double *ego_vs, const double *dt0, int32_t *out_target_lane,
                         int64_t n, void *cuda_stream);

/* LimitSpeed::calculate (src/main.cpp:1068-1150) for one followed car per
 * element, then SpeedController(ego_speed).add_limit_breakpoint (:495-533):
 * out_ls_* = the LimitSpeed result, out_sc_* = the controller's target after
 * the limit, out_flags = PP_F_COLLISION|BRAKE|MAXBRAKE|ADJUST|KEEP. */
int pp_limit_speed_batch(const pp_config *cfg, const double *car_vx, const double *car_vy,
                         const double *next_s, const double *ego_s, const double *ego_speed,
                         const double *ego_acc, const int32_t *in_lane, double *out_ls_speed,
                         double *out_ls_time, double *out_sc_speed, double *out_sc_time,
                         uint32_t *out_flags, int64_t n, void *cuda_stream);

/* TrajectoryBuilder::build (src/main.cpp:565-1049) on explicit inputs: the ego
 * reference point is the last previous point (or ego_x/ego_y when prev_n < 10),
 * sc_* is the SpeedController state handed to build().  prev_x/prev_y [n][10],
 * out_x/out_y [n][50] (NaN beyond out_n), out_flags [n]. */
int pp_trajectory_build_batch(const pp_map *map, const pp_config *cfg, const int32_t *prev_n,
                              const double *prev_x, const double *prev_y, const double *ego_x,
                              const double *ego_y, const double *ego_yaw_deg,
                              const int32_t *target_lane, const double *ego_d,
                              const double *ego_vd, const double *sc_start,
                              const double *sc_target, const double *sc_time, double *out_x,
                              double *out_y, int32_t *out_n, uint32_t *out_flags, int64_t n,
                              void *cuda_stream);

/* The control points of TrajectoryBuilder::build alone (src/main.cpp:638-768), in the map
 * frame, as the reference logs them (control_points=, :779-781): the start point (pos_x,
 * pos_y) = the last kept previous point, or the telemetry pose on a cold start; then up to 5
 * points on the centre line of target_lane.  sc_start = SpeedController::start_speed (the ego
 * speed).  out_x / out_y [n][6] (quiet NaN beyond out_n[n]). */
int pp_control_points_batch(const pp_map *map, const double *pos_x, const double *pos_y,
                            const int32_t *target_lane, const double *ego_d, const double *ego_vd,
                            const double *sc_start, double *out_x, double *out_y, int32_t *out_n,
                            int64_t n, void *cuda_stream);

/* SpeedController (src/main.cpp:488-548) on n explicit controllers
 * (start, target, time, shift [n], all read; target/time/shift may be rewritten):
 *   op 0  get_speed(a)                 -> out[n]            (:503-512)
 *   op 1  add_limit_breakpoint(a, b)   -> target, time      (:513-533)
 *   op 2  override_speed(a, b)         -> shift             (:534-547)
 *   op 3  SpeedController(start)       -> target, time, shift (:493-501; a, b unused)
 * a, b [n] are the method's arguments; out may be NULL for ops 1-3, a/b for op 3. */
int pp_speed_controller_batch(int32_t op, const double *start, double *target, double *time,
                              double *shift, const double *a, const double *b, double *out,
                              int64_t n, void *cuda_stream);

/* Device-memory helpers, so that a caller (and include/pp.hpp) needs neither
 * the CUDA headers nor libcudart of its own: plain cudaMalloc / cudaFree /
 * cudaMemcpy (synchronous) / cudaDeviceSynchronize on the current device. */
int pp_dev_alloc(void **out, size_t bytes);
int pp_dev_free(void *p);
/* Page-locked host memory (cudaHostAlloc / cudaFreeHost): what the buffers handed to
 * pp_plan_batch_host[_split] should live in — copies from pageable memory are staged by the
 * driver and do not overlap with anything. */
int pp_host_alloc(void **out, size_t bytes);
int pp_host_free(void *p);
int pp_dev_upload(void *dst_dev, const void *src_host, size_t bytes);
int pp_dev_download(void *dst_host, const void *src_dev, size_t bytes);
int pp_dev_sync(void);
/* ... and what a host program driving several devices needs (tools/pp_multi.cpp): make a device
 * current for the calling thread, a stream on the current device (cudaStreamNonBlocking). */
int pp_dev_set(int device);
int pp_stream_create(void **stream_out);
int pp_stream_sync(void *stream);
int pp_stream_destroy(void *stream);

/* Device self-test of the exact-arithmetic helpers the kernels use in place of
 * generic divisions / fmod / atan2 (Markstein quotient with cached reciprocal,
 * x/50, angle wrap, small-slope atan): n random trials; counts_dev[8]:
 * [0..2] = number of results that differ bitwise from the generic operation
 * (must be 0), [3] = largest |fast atan - atan2| seen, in ulps, [4..7] = number
 * of results of the emission kernel's unguarded versions (reciprocal, x/50,
 * atan, angle wrap) that differ from the guarded helpers inside the range their
 * "not covered" flag leaves clear (must be 0). */
int pp_selftest_math(int64_t n, uint64_t seed, int64_t *counts_dev, void *cuda_stream);

/* ---- synthetic workload (host; SURVEY §8d config 2/5).  Counter-based RNG
 * keyed by (seed, frame index): any sub-range can be generated on any rank.
 * `out` holds HOST pointers (const is cast away; caller-owned). ---- */
int pp_synth_frames(const pp_map *map, uint64_t seed, int64_t first_frame, int64_t n_frames,
                    int32_t n_cars, int32_t rare_permille, const pp_frames *out);
/* The same frames, bit for bit, written by the GPU into DEVICE buffers (asynchronous on
 * cuda_stream): BASELINE config 5 generates its 64M dense frames in HBM, chunk by chunk. */
int pp_synth_frames_dev(const pp_map *map, uint64_t seed, int64_t first_frame, int64_t n_frames,
                        int32_t n_cars, int32_t rare_permille, const pp_frames *out_dev,
                        void *cuda_stream);

/* ---- candidate sweep (BASELINE config 4; SURVEY §8f-2) --------------------------
 * The reference plans ONE trajectory per frame and notes that "multiple
 * trajectories could be calculated and checked" (README.md:207-208).  The sweep
 * does that: for every frame, PP_SWEEP_CANDS = 3 target lanes x 16 target speeds
 * x 8 target times, each candidate being
 *     SpeedController sc(ego_speed); sc.add_limit_breakpoint(v_i, t_j);
 *     TrajectoryBuilder().build(prev, ..., target_lane = lane, ..., sc)
 * (src/main.cpp:493-533,565-1049) with v_i = i * max_speed / 15, t_j = 0.5 (j + 1) s,
 * candidate index = (lane * 16 + i) * 8 + j.  A candidate is scored on its OUTPUT
 * points P_0..P_{n-1} only (so that the reference's unmodified classes are the
 * oracle), with V_k = (P_{k+1} - P_k) * 50 and A_k = (V_{k+1} - V_k) * 50:
 *     score = |lane - target_lane|                        (target_lane: the planner's own
 *                                                          decision for this frame, :1355-1369)
 *           + (max_speed - mean_k |V_k|) / max_speed
 *           + 0.5 * max(0, max_k |A_k| - maximum_acc)
 * and PP_SWEEP_BAD (1e9) if the builder fell back to the angle-based generator
 * (:848), produced fewer than 3 points, or the score is not a finite number
 * below that (NaN points of a standstill candidate).  The lowest score wins (lowest index on
 * ties) and its trajectory is returned. */
#define PP_SWEEP_LANES 3
#define PP_SWEEP_SPEEDS 16
#define PP_SWEEP_TIMES 8
#define PP_SWEEP_CANDS (PP_SWEEP_LANES * PP_SWEEP_SPEEDS * PP_SWEEP_TIMES)
#define PP_SWEEP_BAD 1e9
typedef struct pp_sweep_out {
  int32_t *best;        /* [N] winning candidate index */
  double *best_score;   /* [N] */
  double *next_x;       /* [N][50] its trajectory (NaN beyond n_points) */
  double *next_y;
  int32_t *n_points;    /* [N] */
  double *scores;       /* [N][PP_SWEEP_CANDS], may be NULL */
} pp_sweep_out;
/* in / out hold DEVICE pointers; asynchronous on cuda_stream. */
int pp_sweep_batch(const pp_map *map, const pp_config *cfg, const pp_frames *in,
                   const pp_sweep_out *out, int64_t n_frames, void *cuda_stream);

/* ---- closed-loop rollouts (BASELINE config 3; SURVEY §8f-1) -----------------
 * R independent ego vehicles, each driving in closed loop against its own
 * planner output and its own synthetic traffic, entirely on the device:
 *
 *   every tick   frame  <- simulator state        (kernel)
 *                plan   <- pp_plan_batch(frame)    (the pipeline above)
 *                state  <- simulator step(plan)    (kernel)
 *
 * The simulator model stands in for the Udacity term-3 simulator the reference
 * was validated against (README.md:12-17); it is defined here, not in the
 * reference, and restated on the CPU in oracle/ for the parity tests:
 *   - the ego is moved to the consume_k-th point of the returned trajectory, the
 *     remaining points become previous_path (src/main.cpp:1248-1249), target_lane
 *     is carried over (:1195);  speed_mph = distance moved / (0.02 k) * 2.237;
 *     yaw stays at its initial value (the planner only reads it on a cold start);
 *   - each car keeps (lane, segment, ratio, speed) and advances along its lane
 *     centre line at constant speed (or, with pp_rollouts_set_traffic, follows the
 *     car ahead: PP_TRAFFIC_IDM below); x, y, vx, vy are derived from that;
 *   - a car whose ego-centred s (as matched by the planner this tick) leaves
 *     [-100, 300] m, or that the planner dropped, is respawned ahead (200-300 m)
 *     if it fell behind, behind (60-100 m) otherwise, in a random lane at
 *     50 +- 10 mph, from a counter-based generator keyed by (seed, rollout, car, tick).
 * All of it is + - * / only, so the CPU restatement is bit-identical. */
typedef struct pp_rollouts pp_rollouts; /* opaque: owns the device state */

/* Host view of the simulator state (caller-owned arrays, R rollouts, C cars). */
typedef struct pp_rollout_state {
  double *ego_x, *ego_y, *ego_yaw_deg, *ego_speed_mph; /* [R] */
  int32_t *path_n;                                     /* [R] unconsumed points of the last plan */
  double *path_x, *path_y;                             /* [R][50] */
  int32_t *target_lane;                                /* [R] */
  int32_t *car_lane, *car_wp;                          /* [R][C] lane, segment end waypoint (0..n-1) */
  double *car_ratio, *car_speed;                       /* [R][C] position along the segment, m/s */
  int64_t tick;                                        /* ticks simulated so far */
} pp_rollout_state;

/* Initial state r = a pure function of (seed, first_rollout + r): ego at rest on a random lane
 * centre (cold start), n_cars cars within [-100, 300] m.  Built on the host, uploaded. */
int pp_rollouts_create(const pp_map *map, int64_t n_rollouts, int32_t n_cars, uint64_t seed,
                       int64_t first_rollout, pp_rollouts **out);
void pp_rollouts_destroy(pp_rollouts *r);
/* n_ticks closed-loop ticks, consume_k (1..40) points per tick; asynchronous on cuda_stream. */
int pp_rollouts_run(pp_rollouts *r, const pp_config *cfg, int64_t n_ticks, int32_t consume_k,
                    void *cuda_stream);
/* lean != 0: the per-tick plans keep only what the simulator and the statistics read (trajectory,
 * n_points, lanes, ref_wp, flags, per-car lane and s); the diagnostics and the other per-car
 * outputs are not written (their pointers in pp_rollouts_last are NULL).  Default: everything. */
int pp_rollouts_set_lean(pp_rollouts *r, int lean);
/* Stream groups a tick is cut into (1..8, at least 4,096 rollouts each; 0 = automatic: up to 8
 * groups of at least 16,384 rollouts).  The result does not depend on it. */
int pp_rollouts_set_groups(pp_rollouts *r, int groups);
/* Device views of the LAST tick's frames and plans (valid until the next run / destroy). */
int pp_rollouts_last(const pp_rollouts *r, pp_frames *frames_dev, pp_plans *plans_dev);
/* Copy the simulator state out (synchronises the device). */
int pp_rollouts_get_state(const pp_rollouts *r, pp_rollout_state *host_out);
/* Sum over all ticks so far of the per-tick pp_stats_batch vectors: stats_dev[PP_STATS_LEN]
 * (device, int64).  The multi-GPU job all-reduces this. */
int pp_rollouts_stats(const pp_rollouts *r, int64_t *stats_dev, void *cuda_stream);

/* ---- incident monitor of the rollouts ----------------------------------------------------
 * The reference was judged by the simulator's "distance without incident" and its acceleration
 * and jerk readouts.  The monitor is the simulator model's own referee, part of the model above,
 * evaluated on the device inside the simulator step; it changes nothing the model computes.
 * Its thresholds are fixed here and do not depend on pp_config (the planner's tunables must not
 * move the referee).  Every operation is IEEE double + - * / and sqrt, left to right, per
 * component, without fused multiply-add, so the CPU restatement is bit-identical.
 *
 * Driven points.  D_0 is the ego's initial pose.  A tick that consumes k points drives through
 * points 0..k-1 of its new plan, which become D_{i+1} .. D_{i+k}; each point is 0.02 s after the
 * one before.  A tick with an empty plan drives no point.
 * Kinematics.  The simulator's own formula is not published; this model takes the windows of
 * the Udacity project description (acceleration = change of the average velocity over 0.2 s,
 * jerk over 1 s):
 *   Vbar_i = (D_i - D_{i-10}) / 0.2      defined for i >= 10
 *   A_i    = (Vbar_i - Vbar_{i-10}) / 0.2 defined for i >= 20
 *   J_i    = (A_i - A_{i-50}) / 1.0      defined for i >= 70
 * and their norms sqrt(x*x + y*y).  over-speed: |Vbar_i| > PP_INC_MAX_SPEED, over-acceleration:
 * |A_i| > PP_INC_MAX_ACC, over-jerk: |J_i| > PP_INC_MAX_JERK, each evaluated at every driven point.
 * Lateral position, once per tick at the tick's last driven point P: the reference waypoint of P
 * is the closest of the rows ref_wp-3 .. ref_wp+3 (ref_wp of this tick's plan; strict <, lowest
 * row wins), completed as Map::init_reference_waypoint does, and (ok, lane, d) is
 * Map::lane_matching(P) from that reference.  The ego is off centre when !ok or
 * |d - 4 (lane + 0.5)| > PP_INC_LANE_TOL; an off-centre count of driven points grows by k per
 * off-centre tick and returns to 0 otherwise.  out-of-lane: that count > PP_INC_OUT_POINTS
 * (3.0 s).  off-road: !ok, d < PP_INC_ROAD_MIN_D or d > PP_INC_ROAD_MAX_D.
 * Collisions, at the end of the tick: the ego at P (its position before the tick when no point
 * was driven) against every car at its advanced (lane, wp, ratio), positioned as the frames
 * position it; t = the car's lane tangent, delta = car - ego.  A pair overlaps when
 * |delta.t| < PP_INC_CAR_HALF_LEN and |delta x t| < PP_INC_CAR_HALF_WIDTH.  A collision is an
 * overlap that BEGINS: the pair did not overlap at the previous positions (the ego of this tick's
 * frame, the car before its advance), so a car placed on top of the ego never counts.
 * collision_front: delta.t > 0, the ego drove into the car.  collision_rear: any other; the
 * traffic of this model never brakes, so a rear collision is the traffic model's doing: it is
 * counted but is NOT an incident for clean_m, first_tick or the incident-free share.
 * Counting.  Every kind is edge-triggered: counted when its condition becomes true (an active
 * bit per kind per rollout), not while it stays true; a collision counts once per tick and side
 * in which some overlap begins.  distance_m = sum |D_i - D_{i-1}| in driving order; clean_m =
 * distance since the last incident (the simulator's "distance without incident"): the step is
 * added, best_clean_m = max(best_clean_m, clean_m), then any incident at that point resets
 * clean_m to 0.  Order within a tick: the driven points in order, then the lateral checks, then
 * the collisions.  first_tick is the rollout's tick counter (0 = its first tick) of the first
 * incident, first_kind the smallest kind counted in that tick. */
#define PP_INC_COLLISION_FRONT 0
#define PP_INC_COLLISION_REAR 1
#define PP_INC_OVER_SPEED 2
#define PP_INC_OVER_ACC 3
#define PP_INC_OVER_JERK 4
#define PP_INC_OUT_OF_LANE 5
#define PP_INC_OFF_ROAD 6
#define PP_INC_KINDS 7
#define PP_INC_MAX_SPEED 22.352    /* m/s = 50 mph */
#define PP_INC_MAX_ACC 10.0        /* m/s^2 */
#define PP_INC_MAX_JERK 10.0       /* m/s^3 */
#define PP_INC_LANE_TOL 1.0        /* m from the lane centre */
#define PP_INC_OUT_POINTS 150      /* driven points off centre (3.0 s) before out-of-lane */
#define PP_INC_ROAD_MIN_D 1.0      /* m */
#define PP_INC_ROAD_MAX_D 11.0     /* m */
#define PP_INC_CAR_HALF_LEN 4.5    /* m along the car's lane */
#define PP_INC_CAR_HALF_WIDTH 2.0  /* m across it */
#define PP_INC_HISTORY 70          /* driven points J_i reaches back */
typedef struct pp_rollout_incidents { /* host arrays, R rollouts; any pointer may be NULL */
  int32_t *count;                     /* [R][PP_INC_KINDS] */
  int64_t *first_tick;                /* [R] tick of the first incident (not rear), -1 none */
  int32_t *first_kind;                /* [R] its kind, -1 none */
  double *distance_m, *clean_m, *best_clean_m; /* [R] */
  double *max_speed, *max_acc, *max_jerk;      /* [R] maxima of the defined |Vbar|, |A|, |J| (0 before) */
} pp_rollout_incidents;
/* Copy the incident record out (synchronises the device). */
int pp_rollouts_get_incidents(const pp_rollouts *r, pp_rollout_incidents *host_out);
/* totals_dev[PP_INC_KINDS + 2] (device, int64, overwritten; asynchronous on cuda_stream): the
 * counts per kind summed over the rollouts, then the number of rollouts with at least one incident
 * (first_tick >= 0), then the driven distance in millimetres, sum of llround(distance_m * 1000).
 * All int64, so a multi-GPU job all-reduces it with ncclSum to the same bits on any GPU count. */
#define PP_INC_TOTAL_ROLLOUTS PP_INC_KINDS
#define PP_INC_TOTAL_MM (PP_INC_KINDS + 1)
#define PP_INC_TOTALS_LEN (PP_INC_KINDS + 2)
int pp_rollouts_incident_totals(const pp_rollouts *r, int64_t *totals_dev, void *cuda_stream);

/* ---- traffic models of the rollouts ------------------------------------------------------
 * PP_TRAFFIC_CONSTANT (the default) is the model above: every car keeps its speed.
 * PP_TRAFFIC_IDM replaces the constant-speed advance of a car that is not respawned by the
 * Intelligent Driver Model (Treiber, Hennecke, Helbing 2000): every car follows the nearest car,
 * or the ego, ahead of it in its lane.  Like the monitor, it is IEEE double + - * / and sqrt,
 * left to right, without fused multiply-add, and its parameters below are fixed, independent of
 * pp_config (the planner's tunables must not move the traffic).
 *
 * Along-lane coordinate.  cum(L, w) = sum of len(i, L) for i = 0 .. w-1 in ascending i (len = the
 * table's lane length, column 10 + L); Lambda_L = cum(L, n).  A car at (L, w, u) sits at
 * S = cum(L, w) + u * len(w, L): the segment from row w-1 to row w, as the frames position it.
 * From follower f to candidate c, Delta = S_c - S_f, reduced into [0, Lambda_L) by at most one
 * addition or subtraction of Lambda_L (+ when Delta < 0, - when Delta >= Lambda_L).  c is AHEAD
 * of f when 0 < Delta < Lambda_L / 2, or Delta == 0 and c's slot is higher; the ego is slot C.
 * The leader is the candidate ahead with the smallest Delta, the lowest slot among equal ones.
 *
 * The ego as a leader, at its position before the tick: bit L of `lanes` is set when the lane
 * match of that position is ok and |d - (4 L + 2)| < PP_TRF_EGO_CORRIDOR (an ego changing lanes
 * is in two), and S_ego[L] = cum(L, wrap(rs.wp)) + rs.ratio[L] * len(rs.wp, L), with (rs, d) the
 * reference and the lane match of the monitor's lateral check at the tick's last driven point
 * (RefState::ratio[L] is measured on the segment from row wp-1 to row wp, the one a car at
 * w = wp sits on).  Tick t stores it and tick t+1 reads it.  Before the first tick it comes from
 * Map::init_reference_waypoint's full search at the initial pose.  Its speed is
 * ego_speed_mph / 2.237 (src/main.cpp:1239) of the frame.
 *
 * Step, synchronous: every car's acceleration is taken from the state of all cars before the
 * tick (a car respawned this tick still counts at its old place), with v its speed and v0 its
 * desired speed:
 *   gap  = max(Delta_leader - PP_INC_CAR_HALF_LEN, PP_TRF_GAP_FLOOR)    (0: the monitor's overlap)
 *   s*   = PP_TRF_MIN_GAP + max(0, v * T + v * (v - v_leader) / (2 * sqrt(a * b)))
 *   q = v / v0, q2 = q * q;  acc = a * (1 - q2 * q2 - (s* / gap) * (s* / gap))   (the last
 *          term is 0 without a leader), then clamped to [-PP_TRF_MAX_DEC, a]
 *   v'   = v + acc * dt, floored at 0;  ds = (v + v') * 0.5 * dt;  dt = 0.02 k as before
 * and the car advances ds along its lane with the constant model's segment carry (u += ds / len,
 * ...).  A respawn draws as before; the drawn speed is the car's v0 and its current speed, and its
 * acc is 0.  Selecting the model sets every car's v0 to its speed and its acc to 0.
 * The incident monitor's definitions do not change. */
#define PP_TRAFFIC_CONSTANT 0       /* constant speed (default) */
#define PP_TRAFFIC_IDM 1            /* Intelligent Driver Model car following */
#define PP_TRF_ACC 1.5              /* m/s^2, maximum acceleration a */
#define PP_TRF_DEC 3.0              /* m/s^2, comfortable deceleration b */
#define PP_TRF_MAX_DEC 9.0          /* m/s^2, clamp on braking */
#define PP_TRF_HEADWAY 1.2          /* s, time headway T */
#define PP_TRF_MIN_GAP 2.0          /* m, standstill gap s0 */
#define PP_TRF_GAP_FLOOR 0.1        /* m, smallest gap the formula is given */
#define PP_TRF_EGO_CORRIDOR 3.0     /* m, |d - lane centre| within which the ego leads a lane
                                       (the reference's "car ahead" corridor, src/main.cpp:1383-1411) */
/* Select the traffic model: before the first tick only (PP_E_ARG afterwards, or for an unknown
 * model).  PP_TRAFFIC_IDM allocates its state and computes the ego's initial lane state. */
int pp_rollouts_set_traffic(pp_rollouts *r, int model);
typedef struct pp_rollout_traffic { /* host arrays; any pointer may be NULL */
  double *car_v0, *car_acc;         /* [R][C] desired speed, last applied acceleration */
  int32_t *ego_lanes;               /* [R] bit L: the ego is a leader in lane L */
  double *ego_s;                    /* [R][3] S_ego per lane */
} pp_rollout_traffic;
/* Copy the IDM state out (synchronises the device); the ego part is what the next tick reads.
 * PP_E_ARG unless PP_TRAFFIC_IDM is selected. */
int pp_rollouts_get_traffic(const pp_rollouts *r, pp_rollout_traffic *host_out);

/* ---- flight recorder of the rollouts -----------------------------------------------------
 * An opt-in observer that keeps, for every rollout, the planner frames of its last W ticks and
 * stops writing them (freezes) at the first tick in which a chosen trigger fires, so that the
 * frames a rollout was given before it failed can be read back and replanned as they are.
 *
 * What is recorded.  Tick t is the rollout's own tick counter before the tick.  Unless the
 * rollout is frozen, tick t writes its frame (the frame the simulator builds for the planner)
 * into slot t % W.  Only the fields that vary are stored: ego_x, ego_y, ego_yaw_deg,
 * ego_speed_mph, prev_n, target_lane_in, prev_x[10], prev_y[10], car_x / car_y / car_vx /
 * car_vy[C], 200 + 32 C bytes a frame; car_id[j] = j and n_cars = C are filled in on read-back.
 * Triggers.  `triggers` is a bit mask.  Bit PP_INC_<kind> fires in tick t when the monitor
 * COUNTS an incident of that kind in tick t (edge-triggered, exactly as it counts); bit
 * PP_REC_NONFINITE fires when the rollout's distance_m is not finite after tick t.  At the end
 * of the first tick t in which a bit of the mask fires, the rollout freezes: trigger_tick = t,
 * trigger_bits = every bit of the mask that fired in tick t.  The window then holds ticks
 * max(0, t - W + 1) .. t; its last frame is the frame whose plan the ego was driving when the
 * trigger fired.  A rollout that never triggers keeps its last W ticks.
 * The recorder is an observer: state, plans, statistics, the incident record and the traffic
 * state do not depend on whether it is on, on W or on the mask.
 * Device memory: R * W * (200 + 32 C) bytes; 65,536 rollouts with W = 256 take 9.8 GB at 12
 * cars and 37.7 GB at 64 cars. */
#define PP_REC_NONFINITE PP_INC_KINDS  /* trigger bit: distance_m is not finite */
#define PP_REC_MAX_WINDOW 1024         /* ticks; out-of-lane needs 150 driven points */
/* Before the first tick only (PP_E_ARG afterwards).  window 0 = off (the default), else
 * 1..PP_REC_MAX_WINDOW; triggers: bits below (1u << (PP_REC_NONFINITE + 1)), else PP_E_ARG.
 * If the allocation fails the recorder is left off and the error returned. */
int pp_rollouts_set_recorder(pp_rollouts *r, int32_t window, uint32_t triggers);
typedef struct pp_rollout_recording { /* host arrays, m rows; any pointer may be NULL */
  int64_t *trigger_tick;              /* [m] tick the rollout froze in, -1: not frozen */
  uint32_t *trigger_bits;             /* [m] bits of the mask that fired then, 0: not frozen */
  int64_t *tick;                      /* [m][W] oldest first; -1: slot not filled */
  int32_t *consume_k;                 /* [m][W] consume_k of that tick, 0: slot not filled */
  /* [m * W] frames in pp_frames layout with max_cars = C: frame (i, j) at i * W + j; the
   * frames of unfilled slots are all 0 */
  double *ego_x, *ego_y, *ego_yaw_deg, *ego_speed_mph, *prev_x, *prev_y;
  double *car_x, *car_y, *car_vx, *car_vy;
  int32_t *prev_n, *target_lane_in, *n_cars, *car_id;
} pp_rollout_recording;
/* Read back the windows of m rollouts (synchronises the device).  rollouts: host, m indices in
 * [0, R); NULL means m == R and row i = rollout i.  PP_E_ARG without a recorder or for an index out
 * of range.  With every frame pointer NULL only the trigger arrays are copied (how a caller finds
 * the rollouts worth fetching). */
int pp_rollouts_get_recording(const pp_rollouts *r, const int64_t *rollouts, int64_t m,
                              pp_rollout_recording *host_out);

/* ---- near-miss (surrogate safety) measures of the rollouts --------------------------------
 * An opt-in observer that measures how close each ego comes to a collision, not only whether it
 * has one: time to collision with the car ahead and the car behind (TTC, Hayward 1972), time
 * headway to the car ahead, their running minima and how long each rollout spends below a set of
 * thresholds (time-exposed TTC, Minderhoud & Bovy 2001).  Evaluated once per tick at the
 * collision check's instant.  Every operation is IEEE double + - * /, left to right, without fused
 * multiply-add, so the CPU restatement is bit-identical.
 *
 * Inputs of a tick.  E = the ego before the tick (this tick's frame); k = the points driven this
 * tick; P = the last driven point, or E when k = 0; the ego's velocity U = (P - E) * 50 / k per
 * component, left to right (U = 0 when k = 0).  Every car j after the advance (a respawned car at
 * its new place): its position C and unit lane tangent t as the collision check takes them, and
 * its speed v after the advance (velocity v t).
 * Geometry per car, with the collision check's expressions:
 *   dx = cx - px;  dy = cy - py;  along = dx*tx + dy*ty;  across = dx*ty - dy*tx;  ut = ux*tx + uy*ty
 * The car is in the ego's path when fabs(across) < PP_INC_CAR_HALF_WIDTH.  A measure is defined
 * only when its condition is true (every comparison with a NaN is false: a non-finite ego defines
 * none):
 *   ahead   in path and along >= PP_INC_CAR_HALF_LEN; gap = along - PP_INC_CAR_HALF_LEN
 *             TTC ahead = gap / w with w = ut - v, when w > 0
 *             time headway = gap / ut, when ut > 0
 *   behind  in path and along <= -PP_INC_CAR_HALF_LEN; gap = -along - PP_INC_CAR_HALF_LEN
 *             TTC behind = gap / w with w = v - ut, when w > 0
 * (an overlapping car is the collision check's business and never a near miss).  The tick's value
 * of each measure is its minimum over the cars, +inf when no car defines it.  Every defined value
 * is >= +0.
 * Record per rollout.  min_ttc_front, min_ttc_rear, min_thw: running minima of the tick values
 * (+inf until first defined); min_ttc_front_tick: the rollout's tick counter at which
 * min_ttc_front was last lowered (strict <), -1 never.  time_hist[m][b]: the tick's weight
 * (k > 0 ? k : 1, in units of 0.02 s, the car model's dt) is added to bin b of measure m when the
 * tick's value lies in [e_{b-1}, e_b), with e = PP_SSM_EDGES and e_{-1} = 0; values >= 8 s and
 * +inf are not counted.  Binning uses comparisons only.
 * The observer changes nothing else: state, plans, statistics, the incident record, the traffic
 * state and the recorder are bit-identical with it on or off.  Device memory: 128 R bytes. */
#define PP_SSM_TTC_FRONT 0
#define PP_SSM_TTC_REAR 1
#define PP_SSM_THW 2
#define PP_SSM_MEASURES 3
#define PP_SSM_BINS 8
#define PP_SSM_EDGES {0.5, 1.0, 1.5, 2.0, 3.0, 4.0, 6.0, 8.0} /* s, upper bin edges */
/* Before the first tick only (PP_E_ARG afterwards).  on != 0 allocates and clears the record;
 * on == 0 (the default) frees it.  If the allocation fails the observer is left off. */
int pp_rollouts_set_surrogate(pp_rollouts *r, int on);
typedef struct pp_rollout_surrogate { /* host arrays, R rollouts; any pointer may be NULL */
  double *min_ttc_front, *min_ttc_rear, *min_thw; /* [R] s, +inf: never defined */
  int64_t *min_ttc_front_tick;                    /* [R] -1: never defined */
  int32_t *time_hist;                             /* [R][PP_SSM_MEASURES][PP_SSM_BINS] */
} pp_rollout_surrogate;
/* Copy the record out (synchronises the device).  PP_E_ARG when the observer is off. */
int pp_rollouts_get_surrogate(const pp_rollouts *r, pp_rollout_surrogate *host_out);
/* totals_dev[PP_SSM_TOTALS_LEN] (device, int64, overwritten; asynchronous on cuda_stream):
 * entry m * PP_SSM_BINS + b is time_hist[.][m][b] summed over the rollouts; entry
 * PP_SSM_TOTAL_MIN + m * PP_SSM_BINS + b is the number of rollouts whose minimum of measure m lies
 * in bin b (binned as above).  All int64, so a multi-GPU job all-reduces it with ncclSum.
 * PP_E_ARG when the observer is off. */
#define PP_SSM_TOTAL_MIN (PP_SSM_MEASURES * PP_SSM_BINS)
#define PP_SSM_TOTALS_LEN (2 * PP_SSM_MEASURES * PP_SSM_BINS)
int pp_rollouts_surrogate_totals(const pp_rollouts *r, int64_t *totals_dev, void *cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* PP_B200_H */
