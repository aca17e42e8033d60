// pp_api.cu — the extern "C" boundary around the kernels: errors, config,
// map lifetime, and the host-buffer entry point (H2D / plan / D2H pipeline).
#include <cuda_runtime.h>

#include <atomic>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "pp_internal.h"

// The planner keeps up to nine streams busy at once (the caller's, four chunk pipes and their
// side streams; a rollouts object: four groups and their side streams).  CUDA maps streams onto
// CUDA_DEVICE_MAX_CONNECTIONS hardware work queues, 8 by default: with more streams than queues
// two independent streams share one and serialise, differently from run to run (the closed-loop
// rollout job measured anywhere between 62 and 217 M ego-frames/s; with 32 queues 200-207 M,
// profiles/probe_connections.sh).  The variable is read when the CUDA context is created, so a
// process that wants the extra queues calls pp_init() before its first CUDA call (or exports the
// variable itself).  The library never touches the environment on its own.
extern "C" int pp_init(void) {
  if (setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0) != 0) return PP_E_ARG;
  return PP_OK;
}

namespace {
std::mutex g_err_mu;
std::string g_err = "";
std::atomic<long long> g_launches{0};
}  // namespace

namespace ppi {

void set_cuda_error(const char *what, int cuda_err, const char *text) {
  std::lock_guard<std::mutex> lk(g_err_mu);
  char buf[512];
  std::snprintf(buf, sizeof buf, "%s: CUDA error %d (%s)", what ? what : "?", cuda_err,
                text ? text : "");
  g_err = buf;
}

void count_launch(int n) { g_launches += n; }

int check_map_device(const pp_map *map, const char *who) {
  if (!map) return PP_E_ARG;
  if (!map->dev_table) {
    set_cuda_error(who, 0, "map has no device table (no usable CUDA device)");
    return PP_E_CUDA;  // there is no CPU planning path
  }
  int dev = -1;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) {
    set_cuda_error("cudaGetDevice", (int)e, cudaGetErrorString(e));
    cudaGetLastError();
    return PP_E_CUDA;
  }
  if (dev != map->device) {
    char msg[160];
    std::snprintf(msg, sizeof msg, "map lives on device %d but device %d is current", map->device,
                  dev);
    set_cuda_error(who, 0, msg);
    return PP_E_ARG;
  }
  return PP_OK;
}

int upload_map(pp_map *m) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) {
    set_cuda_error("cudaGetDevice", (int)e, cudaGetErrorString(e));
    cudaGetLastError();
    return PP_E_CUDA;
  }
  // device copy = the table padded with PPD_PAD wrapped rows at both ends (pp_device.cuh)
  const int pad = 24;
  static_assert(pad == PPD_PAD_ROWS, "padding must match the device code");
  std::vector<double> padded((size_t)(m->n + 2 * pad) * PP_MAP_STRIDE);
  for (int r = 0; r < m->n + 2 * pad; r++) {
    int src = (r - pad) % m->n;
    if (src < 0) src += m->n;
    std::memcpy(&padded[(size_t)r * PP_MAP_STRIDE], &m->table[(size_t)src * PP_MAP_STRIDE],
                PP_MAP_STRIDE * sizeof(double));
  }
  padded.resize(padded.size() + 2, 0.0);  // slack: the kernels stage it in 16-byte granules
  const size_t bytes = padded.size() * sizeof(double);
  e = cudaMalloc(&m->dev_table, bytes);
  if (e != cudaSuccess) {
    m->dev_table = nullptr;
    set_cuda_error("cudaMalloc(map)", (int)e, cudaGetErrorString(e));
    cudaGetLastError();
    return PP_E_CUDA;
  }
  e = cudaMemcpy(m->dev_table, padded.data(), bytes, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    cudaFree(m->dev_table);
    m->dev_table = nullptr;
    set_cuda_error("cudaMemcpy(map)", (int)e, cudaGetErrorString(e));
    cudaGetLastError();
    return PP_E_CUDA;
  }
  e = cudaMalloc(&m->dev_yaw, m->yaw.size() * sizeof(double));
  if (e == cudaSuccess)
    e = cudaMemcpy(m->dev_yaw, m->yaw.data(), m->yaw.size() * sizeof(double), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    cudaFree(m->dev_table);
    if (m->dev_yaw) cudaFree(m->dev_yaw);
    m->dev_table = nullptr;
    m->dev_yaw = nullptr;
    set_cuda_error("cudaMalloc/cudaMemcpy(yaw table)", (int)e, cudaGetErrorString(e));
    cudaGetLastError();
    return PP_E_CUDA;
  }
  m->device = dev;
  return PP_OK;
}

void free_map_device(pp_map *m) {
  if (m && m->dev_table) {
    cudaFree(m->dev_table);
    m->dev_table = nullptr;
  }
  if (m && m->dev_yaw) {
    cudaFree(m->dev_yaw);
    m->dev_yaw = nullptr;
  }
}

}  // namespace ppi

extern "C" {

int pp_version(void) { return PP_VERSION; }

const char *pp_strerror(int code) {
  switch (code) {
    case PP_OK: return "ok";
    case PP_E_ARG: return "invalid argument";
    case PP_E_CUDA: return "CUDA error (see pp_last_cuda_error)";
    case PP_E_IO: return "map file could not be read";
    case PP_E_NOMEM: return "out of memory";
    case PP_E_RANGE: return "size out of range";
    default: return "unknown error";
  }
}

const char *pp_last_cuda_error(void) {
  static thread_local std::string copy;
  std::lock_guard<std::mutex> lk(g_err_mu);
  copy = g_err;
  return copy.c_str();
}

int pp_device_count(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    ppi::set_cuda_error("cudaGetDeviceCount", (int)e, cudaGetErrorString(e));
    cudaGetLastError();
    return PP_E_CUDA;
  }
  return n;
}

int64_t pp_launch_count(void) { return (int64_t)g_launches.load(); }

int pp_config_default(pp_config *cfg) {
  if (!cfg) return PP_E_ARG;
  cfg->relaxed_acc = 5;                    // src/main.cpp:39
  cfg->min_relaxed_acc_while_braking = 4;  // :40
  cfg->maximum_acc = 8;                    // :42
  cfg->max_speed = 22.2;                   // :45
  cfg->car_length = 4.5;                   // :46
  cfg->safety_distance = 2;                // :47
  cfg->keep_distance = 10;                 // :48
  cfg->keep_distance_leeway = 0.5;         // :49
  cfg->test_fast_lane_change = 0;          // :30
  cfg->reserved = 0;
  return PP_OK;
}

// The table is always built on the host.  If no CUDA device is usable the map
// is still returned (so that Map::Init parity and the synthetic generator can
// be exercised on a CPU-only box) but it has no device table and every
// planning call on it fails with PP_E_CUDA.
int pp_map_create(const double *wx, const double *wy, int n, pp_map **out) {
  if (!out) return PP_E_ARG;
  *out = nullptr;
  pp_map *m = new (std::nothrow) pp_map();
  if (!m) return PP_E_NOMEM;
  int rc = ppi::build_map_table(wx, wy, n, m->table);
  if (rc != PP_OK) {
    delete m;
    return rc;
  }
  m->n = n;
  ppi::build_yaw_table(m->table, n, m->yaw);
  ppi::upload_map(m);  // failure is recorded in pp_last_cuda_error(); see above
  *out = m;
  return PP_OK;
}

int pp_map_create_from_csv(const char *path, pp_map **out) {
  if (!out) return PP_E_ARG;
  *out = nullptr;
  std::vector<double> wx, wy;
  int rc = ppi::read_map_csv(path, wx, wy);
  if (rc != PP_OK) return rc;
  return pp_map_create(wx.data(), wy.data(), (int)wx.size(), out);
}

void pp_map_destroy(pp_map *map) {
  if (!map) return;
  ppi::free_map_device(map);
  delete map;
}

int pp_map_num_waypoints(const pp_map *map) { return map ? map->n : PP_E_ARG; }

int pp_map_has_device(const pp_map *map) { return map && map->dev_table ? 1 : 0; }

int pp_map_table(const pp_map *map, double *out) {
  if (!map || !out) return PP_E_ARG;
  std::memcpy(out, map->table.data(), map->table.size() * sizeof(double));
  return PP_OK;
}

#define PP_CK(call, what)                                           \
  do {                                                              \
    cudaError_t e_ = (call);                                        \
    if (e_ != cudaSuccess) {                                        \
      ppi::set_cuda_error(what, (int)e_, cudaGetErrorString(e_));   \
      cudaGetLastError();                                           \
      return PP_E_CUDA;                                             \
    }                                                               \
  } while (0)

int pp_dev_alloc(void **out, size_t bytes) {
  if (!out) return PP_E_ARG;
  *out = nullptr;
  PP_CK(cudaMalloc(out, bytes ? bytes : 1), "pp_dev_alloc");
  return PP_OK;
}
int pp_dev_free(void *p) {
  if (p) PP_CK(cudaFree(p), "pp_dev_free");
  return PP_OK;
}
int pp_host_alloc(void **out, size_t bytes) {
  if (!out) return PP_E_ARG;
  *out = nullptr;
  PP_CK(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault), "pp_host_alloc");
  return PP_OK;
}
int pp_host_free(void *p) {
  if (p) PP_CK(cudaFreeHost(p), "pp_host_free");
  return PP_OK;
}
int pp_dev_upload(void *dst_dev, const void *src_host, size_t bytes) {
  if (bytes && (!dst_dev || !src_host)) return PP_E_ARG;
  if (bytes) PP_CK(cudaMemcpy(dst_dev, src_host, bytes, cudaMemcpyHostToDevice), "pp_dev_upload");
  return PP_OK;
}
int pp_dev_download(void *dst_host, const void *src_dev, size_t bytes) {
  if (bytes && (!dst_host || !src_dev)) return PP_E_ARG;
  if (bytes)
    PP_CK(cudaMemcpy(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost), "pp_dev_download");
  return PP_OK;
}
int pp_dev_sync(void) {
  PP_CK(cudaDeviceSynchronize(), "pp_dev_sync");
  return PP_OK;
}
int pp_dev_set(int device) {
  PP_CK(cudaSetDevice(device), "pp_dev_set");
  return PP_OK;
}
int pp_stream_create(void **stream_out) {
  if (!stream_out) return PP_E_ARG;
  cudaStream_t st = nullptr;
  PP_CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking), "pp_stream_create");
  *stream_out = st;
  return PP_OK;
}
int pp_stream_sync(void *stream) {
  PP_CK(cudaStreamSynchronize((cudaStream_t)stream), "pp_stream_sync");
  return PP_OK;
}
int pp_stream_destroy(void *stream) {
  if (stream) PP_CK(cudaStreamDestroy((cudaStream_t)stream), "pp_stream_destroy");
  return PP_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------
// pp_plan_batch_host: the drop-in for a CPU caller.  Frames are cut into
// chunks; each chunk's inputs go up, are planned, and its plans come back on
// one of kStreams streams, so the H2D copy of chunk c+1, the kernel of chunk c
// and the D2H copy of chunk c-1 overlap.  Device staging buffers are kept per
// thread between calls.
// ---------------------------------------------------------------------------
namespace {

#ifndef PP_HOST_STREAMS
#define PP_HOST_STREAMS 3
#endif
constexpr int kStreams = PP_HOST_STREAMS;
// Chunk schedule: small chunks at both ends (the first chunk's upload and the last chunk's
// download are not overlapped with anything), large ones in the middle (a copy costs ~7 us
// of set-up whatever its size, and every chunk is 37 copies).
constexpr int64_t kChunkFirst = 32768;  // gpurun_out/e2e_sweep.log: 22.3 ms per 1M frames
constexpr int64_t kChunkCap = 131072;    // (the PCIe floor of the box is ~20 ms)

// tuning knobs for experiments (profiles/): PP_HOST_CHUNK_FIRST / PP_HOST_CHUNK_CAP in frames
int64_t env_i64(const char *name, int64_t dflt) {
  const char *v = getenv(name);
  if (!v || !*v) return dflt;
  const long long k = atoll(v);
  return k > 0 ? (int64_t)k : dflt;
}

std::vector<int64_t> chunk_schedule(int64_t n) {
  static const int64_t first = env_i64("PP_HOST_CHUNK_FIRST", kChunkFirst);
  static const int64_t cap = env_i64("PP_HOST_CHUNK_CAP", kChunkCap);
  std::vector<int64_t> head, tail;
  int64_t rem = n, s = first < cap ? first : cap;
  while (rem > 0) {
    const int64_t h = s < rem ? s : rem;
    head.push_back(h);
    rem -= h;
    if (rem <= 0) break;
    const int64_t t = s < rem ? s : rem;
    tail.push_back(t);
    rem -= t;
    if (s < cap) s = s * 2 < cap ? s * 2 : cap;
  }
  head.insert(head.end(), tail.rbegin(), tail.rend());
  return head;
}

struct Field {
  size_t elem;   // bytes per element
  size_t inner;  // elements per frame
};

struct Staging {
  int device = -1;
  int max_cars = -1;
  int64_t cap = 0;
  cudaStream_t streams[kStreams] = {};
  char *in_buf[kStreams] = {};
  char *out_buf[kStreams] = {};
  size_t in_bytes = 0, out_bytes = 0;
  // split rows (pp_plan_batch_host_split): per slot the compact tails [cap][40] x, y; mapped
  // pinned host blocks for the list of frames without kept points and their heads [.][10] x, y
  // of one call (grow-only)
  char *split_buf[kStreams] = {};
  int64_t split_cap = 0;
  int32_t *h_idx = nullptr, *d_idx = nullptr;  // mapped: d_* is the device's view
  double *h_head = nullptr, *d_head = nullptr;
  int64_t h_cap = 0;
  void release_split() {
    for (int i = 0; i < kStreams; i++) {
      if (split_buf[i]) cudaFree(split_buf[i]);
      split_buf[i] = nullptr;
    }
    split_cap = 0;
  }
  void release() {
    release_split();
    for (int i = 0; i < kStreams; i++) {
      if (in_buf[i]) cudaFree(in_buf[i]);
      if (out_buf[i]) cudaFree(out_buf[i]);
      if (streams[i]) cudaStreamDestroy(streams[i]);
      in_buf[i] = out_buf[i] = nullptr;
      streams[i] = nullptr;
    }
    cap = 0;
  }
  ~Staging() {
    release();
    if (h_idx) cudaFreeHost(h_idx);
    if (h_head) cudaFreeHost(h_head);
  }
};

thread_local Staging t_stage;

using ppi::align256;

#define CK(call)                                                    \
  do {                                                              \
    cudaError_t e_ = (call);                                        \
    if (e_ != cudaSuccess) {                                        \
      ppi::set_cuda_error(#call, (int)e_, cudaGetErrorString(e_));  \
      cudaGetLastError();                                           \
      return PP_E_CUDA;                                             \
    }                                                               \
  } while (0)

constexpr int kTailLen = PP_PATH_LEN - PP_PREV_KEEP;

// Split rows, step 1: columns PP_PREV_KEEP.. of the trajectory rows -> compact [n][kTailLen]
// rows (a flat run for the download; a pitched copy of 320-byte rows is a poor DMA shape, see
// below).  One double2 per thread and trip, x and y in the same pass.
__global__ void __launch_bounds__(256)
k_split_tail(const double *__restrict__ nx, const double *__restrict__ ny, int64_t n,
             double *__restrict__ tx, double *__restrict__ ty) {
  constexpr int kPairs = kTailLen / 2;
  const int64_t total = n * kPairs;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / kPairs;
    const int col = (int)(i - row * kPairs);
    const int64_t src = row * (PP_PATH_LEN / 2) + PP_PREV_KEEP / 2 + col;
    reinterpret_cast<double2 *>(tx)[i] = reinterpret_cast<const double2 *>(nx)[src];
    reinterpret_cast<double2 *>(ty)[i] = reinterpret_cast<const double2 *>(ny)[src];
  }
}
static_assert(PP_PATH_LEN % 2 == 0 && PP_PREV_KEEP % 2 == 0, "k_split_tail copies double2");

// Split rows, step 2: the first PP_PREV_KEEP points of the listed frames (those that kept no
// previous points: all 50 of theirs are new) -> compact [k][PP_PREV_KEEP] rows.
__global__ void __launch_bounds__(256)
k_gather_heads(const double *__restrict__ nx, const double *__restrict__ ny,
               const int32_t *__restrict__ idx, int64_t k, double *__restrict__ hx,
               double *__restrict__ hy) {
  const int64_t total = k * PP_PREV_KEEP;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = i / PP_PREV_KEEP;
    const int col = (int)(i - j * PP_PREV_KEEP);
    const int64_t src = (int64_t)idx[j] * PP_PATH_LEN + col;
    hx[i] = nx[src];
    hy[i] = ny[src];
  }
}

// The per-frame scalars (44 of the 636 input bytes, 20 of the 660 output bytes of a frame) do
// not go through the copy engines when the caller's arrays are page-locked: twelve copies of
// 0.5-1 MB per chunk cost the duplex pipeline more than their bytes (profiles/
// r2_pcie_small.log: 17.1 ms per 1M frames with them, 16.0 without, 16.7 with this kernel).
// One launch per chunk and direction moves them between the host arrays, read or written in
// place over PCIe, and the staging buffers.
constexpr int kMoveMax = 18;
struct Move {
  const char *src[kMoveMax];
  char *dst[kMoveMax];
  int bytes[kMoveMax];  // 4 or 8 per element
  int count;
};
constexpr int kMoveBlocks = 64;  // blocks: 16 is too few (18.7 ms), 64 and 296 alike

__global__ void __launch_bounds__(256) k_move_small(const Move p, int64_t n) {
  const int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t step = (int64_t)gridDim.x * blockDim.x;
  for (int f = 0; f < p.count; f++) {
    if (p.bytes[f] == 8) {
      const double *s = reinterpret_cast<const double *>(p.src[f]);
      double *d = reinterpret_cast<double *>(p.dst[f]);
      for (int64_t i = i0; i < n; i += step) d[i] = s[i];
    } else {
      const int32_t *s = reinterpret_cast<const int32_t *>(p.src[f]);
      int32_t *d = reinterpret_cast<int32_t *>(p.dst[f]);
      for (int64_t i = i0; i < n; i += step) d[i] = s[i];
    }
  }
}

// the device's view of a page-locked host pointer, or null when the memory is pageable (or
// the array is not aligned to its elements: such a caller gets the copy engine)
char *mapped_view(const void *host, size_t elem) {
  if (!host || ((uintptr_t)host & (elem - 1)) != 0) return nullptr;
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, host) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return a.type == cudaMemoryTypeHost ? (char *)a.devicePointer : nullptr;
}

int plan_host(const pp_map *map, const pp_config *cfg, const pp_frames *in, const pp_plans *out,
              const pp_split_rows *split, int64_t n_frames) {
  if (!map || !cfg || !in || !out || n_frames < 0) return PP_E_ARG;
  if (split) {  // the trajectories come back in two parts instead of whole rows
    if (!split->head_x || !split->head_y || !split->tail_x || !split->tail_y) return PP_E_ARG;
    if (out->next_x || out->next_y) return PP_E_ARG;
  }
  if (!map->dev_table) {
    ppi::set_cuda_error("pp_plan_batch_host: map has no device table (no usable CUDA device)", 0,
                        "");
    return PP_E_CUDA;
  }
  {
    const int rc = ppi::check_map_device(map, "pp_plan_batch_host");
    if (rc != PP_OK) return rc;
  }
  if (in->max_cars < 0 || in->max_cars > PP_MAX_CARS) return PP_E_RANGE;
  if (n_frames == 0) return PP_OK;
  const size_t mc = (size_t)in->max_cars;

  // field tables: (host pointer, bytes per frame), in struct order
  struct HIn { const void *p; size_t bpf; };
  const bool frozen = in->car_frozen_lane != nullptr;
  if (frozen && (!in->car_frozen_s || !in->car_frozen_d || !in->car_frozen_vs || !in->car_frozen_vd))
    return PP_E_ARG;
  constexpr int kIn = 19;
  const HIn hin[kIn] = {
      {in->ego_x, 8}, {in->ego_y, 8}, {in->ego_yaw_deg, 8}, {in->ego_speed_mph, 8},
      {in->prev_n, 4}, {in->prev_x, 8 * PP_PREV_KEEP}, {in->prev_y, 8 * PP_PREV_KEEP},
      {in->target_lane_in, 4}, {in->n_cars, 4}, {in->car_id, 4 * mc}, {in->car_x, 8 * mc},
      {in->car_y, 8 * mc}, {in->car_vx, 8 * mc}, {in->car_vy, 8 * mc},
      {in->car_frozen_lane, 4 * mc}, {in->car_frozen_s, 8 * mc}, {in->car_frozen_d, 8 * mc},
      {in->car_frozen_vs, 8 * mc}, {in->car_frozen_vd, 8 * mc}};
  struct HOut { void *p; size_t bpf; };
  const HOut hout[23] = {
      {out->next_x, 8 * PP_PATH_LEN}, {out->next_y, 8 * PP_PATH_LEN}, {out->n_points, 4},
      {out->ego_lane, 4}, {out->ref_wp, 4}, {out->target_lane, 4}, {out->flags, 4},
      {out->ego_s, 8}, {out->ego_d, 8}, {out->ego_vs, 8}, {out->ego_vd, 8}, {out->ego_speed, 8},
      {out->ego_acc, 8}, {out->target_speed, 8}, {out->target_time, 8}, {out->next_car_id, 4},
      {out->next_car_in_target_lane, 4}, {out->car_s, 8 * mc}, {out->car_d, 8 * mc},
      {out->car_vs, 8 * mc}, {out->car_vd, 8 * mc}, {out->car_lane, 4 * mc},
      {out->car_next_wp, 4 * mc}};
  for (int i = 0; i < 9; i++)
    if (!hin[i].p) return PP_E_ARG;
  if (mc > 0)
    for (int i = 9; i < 14; i++)
      if (!hin[i].p) return PP_E_ARG;
  for (int i = split ? 2 : 0; i < 7; i++)
    if (!hout[i].p) return PP_E_ARG;

  int dev = 0;
  CK(cudaGetDevice(&dev));
  Staging &sg = t_stage;
  const std::vector<int64_t> sizes = chunk_schedule(n_frames);
  int64_t chunk = 0;  // staging capacity = the largest chunk of the schedule
  for (int64_t v : sizes) chunk = v > chunk ? v : chunk;
  size_t in_bpf = 0, out_bpf = 0;
  for (int i = 0; i < kIn; i++) in_bpf += align256(hin[i].bpf * (size_t)chunk);
  for (int i = 0; i < 23; i++) out_bpf += align256(hout[i].bpf * (size_t)chunk);
  if (sg.device != dev || sg.max_cars != in->max_cars || sg.cap < chunk || sg.in_bytes < in_bpf) {
    sg.release();
    for (int i = 0; i < kStreams; i++) {
      CK(cudaStreamCreateWithFlags(&sg.streams[i], cudaStreamNonBlocking));
      CK(cudaMalloc(&sg.in_buf[i], in_bpf));
      CK(cudaMalloc(&sg.out_buf[i], out_bpf));
    }
    sg.device = dev;
    sg.max_cars = in->max_cars;
    sg.cap = chunk;
    sg.in_bytes = in_bpf;
    sg.out_bytes = out_bpf;
  }
  // split rows: which frames kept no previous points is known from the caller's prev_n (the
  // rule of ego_state, src/main.cpp:1261), so the lists are built here, on the host
  int64_t n_short = 0;
  if (split) {
    if (sg.split_cap < sg.cap) {
      sg.release_split();
      const size_t c = (size_t)sg.cap;
      const size_t bytes = 2 * align256(c * kTailLen * 8);
      for (int i = 0; i < kStreams; i++) CK(cudaMalloc(&sg.split_buf[i], bytes));
      sg.split_cap = sg.cap;
    }
  }
  // the scalars that can bypass the copy engines (PP_HOST_NO_ZERO_COPY: never)
  static const bool zero_copy = getenv("PP_HOST_NO_ZERO_COPY") == nullptr;
  char *min_view[kIn] = {}, *mout_view[23] = {};
  if (zero_copy) {
    for (int i : {0, 1, 2, 3, 4, 7, 8}) min_view[i] = mapped_view(hin[i].p, hin[i].bpf);
    for (int i = 2; i < 17; i++) mout_view[i] = mapped_view(hout[i].p, hout[i].bpf);
  }

  // (Measured and dropped, profiles/bench_r2b_n1_{pitched,flat}_d2h.json: bringing down only the
  // 40 new columns of a trajectory with a pitched copy — the 10 kept ones are the caller's own
  // previous points — and filling the rest on the host moves 17 % fewer bytes but runs at
  // 44.7 M frames/s against 52.3 M for whole rows: 320-byte rows are a poor DMA shape.  The
  // split-rows entry point compacts the new columns on the device instead.)
  // Nothing may still be writing into the caller's buffers when this returns, whatever the
  // outcome: a failure below joins the streams before it reports.
  struct Join {
    Staging &sg;
    ~Join() {
      for (int i = 0; i < kStreams; i++)
        if (sg.streams[i]) cudaStreamSynchronize(sg.streams[i]);
      cudaGetLastError();
    }
  } join_on_exit{sg};
  // experiments only (profiles/r2_e2e_parts.log): leave out the uploads (1), the kernels (2)
  // or the downloads (4) to see what each part of the pipeline costs
  static const int64_t probe = env_i64("PP_HOST_PROBE", 0);
  int slot = 0;
  int64_t lo = 0;
  int64_t short_done = 0;  // entries of h_idx / h_head used by the chunks so far
  std::vector<int64_t> short_of(sizes.size(), 0);
  int sms = 148;
  if (split && cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
    cudaGetLastError();
    sms = 148;
  }
  for (size_t ci = 0; ci < sizes.size(); lo += sizes[ci], ci++, slot = (slot + 1) % kStreams) {
    const int64_t cnt = sizes[ci];
    cudaStream_t st = sg.streams[slot];
    // device-side views of this slot's staging buffers
    const void *din[kIn];
    void *dout[23];
    size_t off = 0;
    for (int i = 0; i < kIn; i++) {
      din[i] = sg.in_buf[slot] + off;
      off += align256(hin[i].bpf * (size_t)sg.cap);
    }
    off = 0;
    for (int i = 0; i < 23; i++) {
      dout[i] = (hout[i].p || i < 2) ? (void *)(sg.out_buf[slot] + off) : nullptr;
      off += align256(hout[i].bpf * (size_t)sg.cap);
    }
    Move mv;
    mv.count = 0;
    for (int i = 0; i < kIn; i++) {
      if (!hin[i].p || hin[i].bpf == 0 || (probe & 1)) continue;
      if (min_view[i]) {
        mv.src[mv.count] = min_view[i] + hin[i].bpf * (size_t)lo;
        mv.dst[mv.count] = (char *)din[i];
        mv.bytes[mv.count++] = (int)hin[i].bpf;
        continue;
      }
      CK(cudaMemcpyAsync((void *)din[i], (const char *)hin[i].p + hin[i].bpf * (size_t)lo,
                         hin[i].bpf * (size_t)cnt, cudaMemcpyHostToDevice, st));
    }
    if (mv.count) {
      k_move_small<<<kMoveBlocks, 256, 0, st>>>(mv, cnt);
      ppi::count_launch(1);
    }
    if (split && ci == 0) {
      // How many frames kept nothing, for the size of the pinned lists: counted while the first
      // chunk's upload is under way.
      for (int64_t f = 0; f < n_frames; f++) n_short += in->prev_n[f] < PP_PREV_KEEP;
      if (n_short > sg.h_cap) {
        if (sg.h_idx) cudaFreeHost(sg.h_idx);
        if (sg.h_head) cudaFreeHost(sg.h_head);
        sg.h_idx = nullptr;
        sg.h_head = nullptr;
        sg.h_cap = 0;
        sg.d_idx = nullptr;
        sg.d_head = nullptr;
        CK(cudaHostAlloc((void **)&sg.h_idx, (size_t)n_short * 4, cudaHostAllocMapped));
        CK(cudaHostAlloc((void **)&sg.h_head, (size_t)n_short * 2 * PP_PREV_KEEP * 8,
                         cudaHostAllocMapped));
        CK(cudaHostGetDevicePointer((void **)&sg.d_idx, sg.h_idx, 0));
        CK(cudaHostGetDevicePointer((void **)&sg.d_head, sg.h_head, 0));
        sg.h_cap = n_short;
      }
    }
    pp_frames fin;
    fin.ego_x = (const double *)din[0];
    fin.ego_y = (const double *)din[1];
    fin.ego_yaw_deg = (const double *)din[2];
    fin.ego_speed_mph = (const double *)din[3];
    fin.prev_n = (const int32_t *)din[4];
    fin.prev_x = (const double *)din[5];
    fin.prev_y = (const double *)din[6];
    fin.target_lane_in = (const int32_t *)din[7];
    fin.n_cars = (const int32_t *)din[8];
    fin.car_id = (const int32_t *)din[9];
    fin.car_x = (const double *)din[10];
    fin.car_y = (const double *)din[11];
    fin.car_vx = (const double *)din[12];
    fin.car_vy = (const double *)din[13];
    fin.max_cars = in->max_cars;
    fin.reserved = 0;
    fin.car_frozen_lane = frozen ? (const int32_t *)din[14] : nullptr;
    fin.car_frozen_s = frozen ? (const double *)din[15] : nullptr;
    fin.car_frozen_d = frozen ? (const double *)din[16] : nullptr;
    fin.car_frozen_vs = frozen ? (const double *)din[17] : nullptr;
    fin.car_frozen_vd = frozen ? (const double *)din[18] : nullptr;
    pp_plans fout;
    fout.next_x = (double *)dout[0];
    fout.next_y = (double *)dout[1];
    fout.n_points = (int32_t *)dout[2];
    fout.ego_lane = (int32_t *)dout[3];
    fout.ref_wp = (int32_t *)dout[4];
    fout.target_lane = (int32_t *)dout[5];
    fout.flags = (uint32_t *)dout[6];
    fout.ego_s = (double *)dout[7];
    fout.ego_d = (double *)dout[8];
    fout.ego_vs = (double *)dout[9];
    fout.ego_vd = (double *)dout[10];
    fout.ego_speed = (double *)dout[11];
    fout.ego_acc = (double *)dout[12];
    fout.target_speed = (double *)dout[13];
    fout.target_time = (double *)dout[14];
    fout.next_car_id = (int32_t *)dout[15];
    fout.next_car_in_target_lane = (int32_t *)dout[16];
    fout.car_s = (double *)dout[17];
    fout.car_d = (double *)dout[18];
    fout.car_vs = (double *)dout[19];
    fout.car_vd = (double *)dout[20];
    fout.car_lane = (int32_t *)dout[21];
    fout.car_next_wp = (int32_t *)dout[22];
    int rc = (probe & 2) ? PP_OK : pp_plan_batch(map, cfg, &fin, &fout, cnt, st);
    if (rc != PP_OK) return rc;
    if (probe & 4) continue;
    if (split) {
      const size_t c = (size_t)sg.split_cap;
      char *sb = sg.split_buf[slot];
      double *d_tx = (double *)sb;
      double *d_ty = (double *)(sb + align256(c * kTailLen * 8));
      k_split_tail<<<sms * 8, 256, 0, st>>>(fout.next_x, fout.next_y, cnt, d_tx, d_ty);
      ppi::count_launch(1);
      CK(cudaMemcpyAsync(split->tail_x + (size_t)lo * kTailLen, d_tx, (size_t)cnt * kTailLen * 8,
                         cudaMemcpyDeviceToHost, st));
      CK(cudaMemcpyAsync(split->tail_y + (size_t)lo * kTailLen, d_ty, (size_t)cnt * kTailLen * 8,
                         cudaMemcpyDeviceToHost, st));
      // this chunk's frames without kept points: the kernel reads the (chunk-local) index list
      // from the pinned host block and writes the heads into it, in place over PCIe
      int64_t k = 0;
      int32_t *list = sg.h_idx + short_done;
      for (int64_t f = 0; f < cnt; f++)
        if (in->prev_n[lo + f] < PP_PREV_KEEP) list[k++] = (int32_t)f;
      if (k > 0) {
        double *hh = sg.d_head + (size_t)short_done * 2 * PP_PREV_KEEP;
        const int64_t want = (k * PP_PREV_KEEP + 255) / 256;
        k_gather_heads<<<(int)(want < kMoveBlocks ? want : kMoveBlocks), 256, 0, st>>>(
            fout.next_x, fout.next_y, sg.d_idx + short_done, k, hh, hh + (size_t)k * PP_PREV_KEEP);
        ppi::count_launch(1);
        short_done += k;
        short_of[ci] = k;
      }
    }
    mv.count = 0;
    for (int i = 0; i < 23; i++) {
      if (!hout[i].p || hout[i].bpf == 0) continue;
      if (mout_view[i]) {
        mv.src[mv.count] = (const char *)dout[i];
        mv.dst[mv.count] = mout_view[i] + hout[i].bpf * (size_t)lo;
        mv.bytes[mv.count++] = (int)hout[i].bpf;
        continue;
      }
      CK(cudaMemcpyAsync((char *)hout[i].p + hout[i].bpf * (size_t)lo, dout[i],
                         hout[i].bpf * (size_t)cnt, cudaMemcpyDeviceToHost, st));
    }
    if (mv.count) {
      k_move_small<<<kMoveBlocks, 256, 0, st>>>(mv, cnt);
      ppi::count_launch(1);
    }
  }
  for (int i = 0; i < kStreams; i++) CK(cudaStreamSynchronize(sg.streams[i]));
  if (split && n_short > 0) {  // the gathered heads into their rows (80 bytes each, few frames)
    int64_t used = 0, base = 0;
    for (size_t ci = 0; ci < sizes.size(); base += sizes[ci], ci++) {
      const int64_t k = short_of[ci];
      const int32_t *list = sg.h_idx + used;
      const double *hx = sg.h_head + (size_t)used * 2 * PP_PREV_KEEP;
      const double *hy = hx + (size_t)k * PP_PREV_KEEP;
      for (int64_t j = 0; j < k; j++) {
        const size_t row = (size_t)(base + list[j]) * PP_PREV_KEEP;
        std::memcpy(split->head_x + row, hx + (size_t)j * PP_PREV_KEEP, PP_PREV_KEEP * 8);
        std::memcpy(split->head_y + row, hy + (size_t)j * PP_PREV_KEEP, PP_PREV_KEEP * 8);
      }
      used += k;
    }
  }
  return PP_OK;
}

}  // namespace

extern "C" int pp_plan_batch_host(const pp_map *map, const pp_config *cfg, const pp_frames *in,
                                  const pp_plans *out, int64_t n_frames) {
  return plan_host(map, cfg, in, out, nullptr, n_frames);
}

extern "C" int pp_plan_batch_host_split(const pp_map *map, const pp_config *cfg,
                                        const pp_frames *in, const pp_plans *out,
                                        const pp_split_rows *rows, int64_t n_frames) {
  if (!rows) return PP_E_ARG;
  return plan_host(map, cfg, in, out, rows, n_frames);
}
