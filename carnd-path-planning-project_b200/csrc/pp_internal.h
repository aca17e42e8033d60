// Internal declarations shared by the translation units of libpp_b200.so.
#pragma once
#include <cstddef>
#include <cstdint>
#include <vector>

#include "../../include/pp.h"

// rows of wrap-around padding on either side of the device copy of the table
#define PPD_PAD_ROWS 24

struct pp_map {
  int n = 0;                  // waypoints
  std::vector<double> table;  // n * PP_MAP_STRIDE, host copy (row layout of pp.h)
  double *dev_table = nullptr;  // device copy, padded (nullptr if no CUDA device was usable)
  int device = -1;              // CUDA device the table lives on
  std::vector<double> yaw;      // [n][3] lane-segment headings in degrees (synthetic generator)
  double *dev_yaw = nullptr;
};

namespace ppi {

// Host-side Map::Init (reference src/main.cpp:89-131): fills `table`.
int build_map_table(const double *wx, const double *wy, int n, std::vector<double> &table);
// atan2 of every lane segment's direction, in degrees (pp_synth.cu).
void build_yaw_table(const std::vector<double> &table, int n, std::vector<double> &yaw);
// CSV reader with the reference's parsing (src/main.cpp:1171-1191).
int read_map_csv(const char *path, std::vector<double> &wx, std::vector<double> &wy);

// Upload (pp_api.cu).  Returns PP_OK or PP_E_CUDA.
int upload_map(pp_map *m);
void free_map_device(pp_map *m);

void set_cuda_error(const char *what, int cuda_err, const char *text);
// PP_OK when the map's device table lives on the CURRENT device; PP_E_CUDA when the map has no
// device table, PP_E_ARG when it was created on another device (using it would dereference a
// foreign device pointer inside a kernel and poison the context).
int check_map_device(const pp_map *map, const char *who);

// Device buffers are carved into sub-buffers that start on 256-byte boundaries.
inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// Typed sub-buffers of one allocation.  A layout is one block of take() calls run twice: on a
// Carve without a base it only adds up the size (and hands out nullptr), on the allocated base
// it binds the pointers at the same offsets.
struct Carve {
  char *base = nullptr;
  size_t size = 0;  // bytes taken so far, a multiple of 256
  explicit Carve(char *b = nullptr) : base(b) {}
  template <class T>
  void take(T *&p, size_t count) {
    p = base ? (T *)(base + size) : nullptr;
    size += align256(count * sizeof(T));
  }
};

// pp_plan.cu: the pipeline with caller-owned scratch (see there)
size_t plan_scratch_bytes(int64_t n_frames, int max_cars);
// xsum_add (used when stats_dev is null): the pipeline's kernels ADD the checksum of the
// trajectories they write (PP_STAT_XSUM) to *xsum_add, nothing is cleared; honoured only when
// plan_adds_checksum(n_frames) — the single-kernel paths of small batches do not take it.
int plan_batch_scratch(const pp_map *map, const pp_config *cfg, const pp_frames *in,
                       const pp_plans *out, int64_t n_frames, void *cuda_stream,
                       char *caller_scratch, int64_t *stats_dev,
                       unsigned long long *xsum_add = nullptr);
bool plan_adds_checksum(int64_t n_frames);

// pp_frames / pp_plans advanced by `lo` frames
inline pp_frames offset_frames(const pp_frames &a, int64_t lo) {
  pp_frames r = a;
  const int64_t mc = a.max_cars;
  r.ego_x += lo;
  r.ego_y += lo;
  r.ego_yaw_deg += lo;
  r.ego_speed_mph += lo;
  r.prev_n += lo;
  r.prev_x += lo * PP_PREV_KEEP;
  r.prev_y += lo * PP_PREV_KEEP;
  r.target_lane_in += lo;
  r.n_cars += lo;
  if (r.car_id) r.car_id += lo * mc;
  if (r.car_x) r.car_x += lo * mc;
  if (r.car_y) r.car_y += lo * mc;
  if (r.car_vx) r.car_vx += lo * mc;
  if (r.car_vy) r.car_vy += lo * mc;
  if (r.car_frozen_lane) {
    r.car_frozen_lane += lo * mc;
    r.car_frozen_s += lo * mc;
    r.car_frozen_d += lo * mc;
    r.car_frozen_vs += lo * mc;
    r.car_frozen_vd += lo * mc;
  }
  return r;
}
template <class T>
inline void adv(T *&p, int64_t k) {
  if (p) p += k;
}
inline pp_plans offset_plans(const pp_plans &a, int64_t lo, int64_t mc) {
  pp_plans r = a;
  adv(r.next_x, lo * PP_PATH_LEN);
  adv(r.next_y, lo * PP_PATH_LEN);
  adv(r.n_points, lo);
  adv(r.ego_lane, lo);
  adv(r.ref_wp, lo);
  adv(r.target_lane, lo);
  adv(r.flags, lo);
  adv(r.ego_s, lo);
  adv(r.ego_d, lo);
  adv(r.ego_vs, lo);
  adv(r.ego_vd, lo);
  adv(r.ego_speed, lo);
  adv(r.ego_acc, lo);
  adv(r.target_speed, lo);
  adv(r.target_time, lo);
  adv(r.next_car_id, lo);
  adv(r.next_car_in_target_lane, lo);
  adv(r.car_s, lo * mc);
  adv(r.car_d, lo * mc);
  adv(r.car_vs, lo * mc);
  adv(r.car_vd, lo * mc);
  adv(r.car_lane, lo * mc);
  adv(r.car_next_wp, lo * mc);
  return r;
}


void count_launch(int n = 1);

}  // namespace ppi
