// pp.hpp — C++ host façade over the C ABI of include/pp.h.
//
// Keeps the reference's class and function names as the API surface
// (Fable3/CarND-Path-Planning-Project: src/helpers.h, src/main.cpp, src/spline.h)
// so that host code written against the reference reads the same here:
//
//   reference                                  here (namespace pp)
//   ------------------------------------------------------------------------------
//   Point, distance, distancesq_pt_seg         Point, distance, distancesq_pt_seg      helpers.h:38-40,160-249
//   ClosestWaypoint/NextWaypoint/getFrenet/getXY  same names                           helpers.h:43-155
//   Car (+predicted_s/d)                       Car                                     main.cpp:51-71
//   Map::Init / init_reference_waypoint /      Map (same members; the per-frame        main.cpp:73-358
//     lane_matching / get_lane_pos /             reference_waypoint_* state is kept on
//     project_speed / get_lane_length            the object exactly like the reference)
//   LaneChangePlanner::calculate_target_lane   LaneChangePlanner                       main.cpp:361-485
//   SpeedController                            SpeedController                         main.cpp:488-548
//   LimitSpeed::calculate                      LimitSpeed                              main.cpp:1052-1151
//   TrajectoryBuilder::build                   TrajectoryBuilder                       main.cpp:550-1049
//   tk::spline set_points / operator()         tk::spline                              spline.h:284-396
//   the onMessage planning step                Planner::plan (batch of frames)         main.cpp:1254-1457
//
// Every method that computes something calls the sm_100a kernels through the
// extern "C" layer; there is no CPU planning path behind these classes (a
// process without a usable CUDA device gets pp::Error from the first call).
// The per-object methods move one element through the GPU per call — they exist
// for API parity and for tests; throughput comes from Planner::plan, which hands
// whole SoA frame batches to pp_plan_batch_host / pp_plan_batch.
//
// Header-only, C++11, needs only pp.h and libpp_b200.so (no CUDA headers).
#ifndef PP_B200_HPP
#define PP_B200_HPP

#include <cmath>
#include <cstring>
#include <map>
#include <stdexcept>
#include <string>
#include <vector>

#include "pp.h"

namespace pp {

struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string &what) : std::runtime_error(what), code(c) {}
};

inline void check(int rc, const char *what) {
  if (rc == PP_OK) return;
  std::string msg = std::string(what) + ": " + pp_strerror(rc);
  if (rc == PP_E_CUDA) msg += std::string(" — ") + pp_last_cuda_error();
  throw Error(rc, msg);
}

// Tunables: the reference's globals (src/main.cpp:30,39-49).
inline pp_config default_config() {
  pp_config c;
  check(pp_config_default(&c), "pp_config_default");
  return c;
}

namespace detail {
// A typed device buffer (RAII over pp_dev_alloc / pp_dev_free).
template <class T>
class Dev {
 public:
  explicit Dev(size_t n) : n_(n) { check(pp_dev_alloc(&p_, n * sizeof(T)), "pp_dev_alloc"); }
  Dev(const T *host, size_t n) : n_(n) {
    check(pp_dev_alloc(&p_, n * sizeof(T)), "pp_dev_alloc");
    check(pp_dev_upload(p_, host, n * sizeof(T)), "pp_dev_upload");
  }
  explicit Dev(const std::vector<T> &v) : Dev(v.data(), v.size()) {}
  ~Dev() { pp_dev_free(p_); }
  Dev(const Dev &) = delete;
  Dev &operator=(const Dev &) = delete;
  Dev(Dev &&o) noexcept : p_(o.p_), n_(o.n_) { o.p_ = nullptr; }
  T *get() { return static_cast<T *>(p_); }
  const T *get() const { return static_cast<const T *>(p_); }
  void to_host(T *out) const { check(pp_dev_download(out, p_, n_ * sizeof(T)), "pp_dev_download"); }
  std::vector<T> to_host() const {
    std::vector<T> v(n_);
    if (n_) to_host(v.data());
    return v;
  }
  T first() const {
    T v;
    check(pp_dev_download(&v, p_, sizeof(T)), "pp_dev_download");
    return v;
  }

 private:
  void *p_ = nullptr;
  size_t n_;
};
inline Dev<double> one(double v) { return Dev<double>(&v, 1); }
}  // namespace detail

// ---- helpers.h ---------------------------------------------------------------
struct Point {  // src/helpers.h:160-181 (a value type; no planning arithmetic lives here)
  double x, y;
  Point() : x(0), y(0) {}
  Point(double _x, double _y) : x(_x), y(_y) {}
  Point operator-(const Point B) const { return Point(x - B.x, y - B.y); }
  Point operator+(const Point B) const { return Point(x + B.x, y + B.y); }
  double length() const { return std::sqrt(x * x + y * y); }
  double lengthsq() const { return x * x + y * y; }
  double dotp(Point B) const { return x * B.x + y * B.y; }
};
inline double distance(double x1, double y1, double x2, double y2) {  // src/helpers.h:38-40
  return std::sqrt((x2 - x1) * (x2 - x1) + (y2 - y1) * (y2 - y1));
}

// src/helpers.h:188-249 (same out-parameter order)
inline double distancesq_pt_seg(Point p, Point A, Point B, double &_rnom, double &_rdenom,
                                double &_snom) {
  using detail::one;
  detail::Dev<double> px = one(p.x), py = one(p.y), ax = one(A.x), ay = one(A.y), bx = one(B.x),
                      by = one(B.y);
  detail::Dev<double> d2(1), rn(1), rd(1), sn(1);
  check(pp_distancesq_pt_seg_batch(px.get(), py.get(), ax.get(), ay.get(), bx.get(), by.get(),
                                   d2.get(), rn.get(), rd.get(), sn.get(), 1, nullptr),
        "pp_distancesq_pt_seg_batch");
  _rnom = rn.first();
  _rdenom = rd.first();
  _snom = sn.first();
  return d2.first();
}

// Udacity starter helpers, src/helpers.h:43-155 (never called by the planner).
inline int ClosestWaypoint(double x, double y, const std::vector<double> &maps_x,
                           const std::vector<double> &maps_y) {
  detail::Dev<double> dx = detail::one(x), dy = detail::one(y), mx(maps_x), my(maps_y);
  detail::Dev<int32_t> out(1);
  check(pp_closest_waypoint_batch(dx.get(), dy.get(), mx.get(), my.get(), (int32_t)maps_x.size(),
                                  out.get(), 1, nullptr),
        "pp_closest_waypoint_batch");
  return out.first();
}
inline int NextWaypoint(double x, double y, double theta, const std::vector<double> &maps_x,
                        const std::vector<double> &maps_y) {
  detail::Dev<double> dx = detail::one(x), dy = detail::one(y), dt = detail::one(theta), mx(maps_x),
                      my(maps_y);
  detail::Dev<int32_t> out(1);
  check(pp_next_waypoint_batch(dx.get(), dy.get(), dt.get(), mx.get(), my.get(),
                               (int32_t)maps_x.size(), out.get(), 1, nullptr),
        "pp_next_waypoint_batch");
  return out.first();
}
inline std::vector<double> getFrenet(double x, double y, double theta,
                                     const std::vector<double> &maps_x,
                                     const std::vector<double> &maps_y) {
  detail::Dev<double> dx = detail::one(x), dy = detail::one(y), dt = detail::one(theta), mx(maps_x),
                      my(maps_y), os(1), od(1);
  check(pp_get_frenet_batch(dx.get(), dy.get(), dt.get(), mx.get(), my.get(),
                            (int32_t)maps_x.size(), os.get(), od.get(), 1, nullptr),
        "pp_get_frenet_batch");
  return {os.first(), od.first()};
}
inline std::vector<double> getXY(double s, double d, const std::vector<double> &maps_s,
                                 const std::vector<double> &maps_x,
                                 const std::vector<double> &maps_y) {
  detail::Dev<double> ds = detail::one(s), dd = detail::one(d), ms(maps_s), mx(maps_x), my(maps_y),
                      ox(1), oy(1);
  check(pp_get_xy_batch(ds.get(), dd.get(), ms.get(), mx.get(), my.get(), (int32_t)maps_x.size(),
                        ox.get(), oy.get(), 1, nullptr),
        "pp_get_xy_batch");
  return {ox.first(), oy.first()};
}

// ---- main.cpp ------------------------------------------------------------------
struct Car {  // src/main.cpp:51-71
  int id = 0;
  double x = 0, y = 0, vx = 0, vy = 0;  // input
  double s = 0, d = 0;                  // calculated
  double acc_x = 0, acc_y = 0;
  double vs = 0, vd = 0;
  int lane = 0;
  // not in the reference: this entry was NOT in the current message; the reference still holds
  // it in its persistent map with the s, d, vs, vd, lane of its last sighting (:1194,1325-1334)
  bool frozen = false;
  double predicted_s(double delta_t) const { return s + vs * delta_t; }
  double predicted_d(double delta_t) const { return d + vd * delta_t; }
};

class Map {  // src/main.cpp:73-358
 public:
  struct Waypoint {  // :76-82 (len is declared and never set by the reference either)
    Point ref;
    Point lane_center[PP_NUM_LANES];
    double len;
    double nx, ny;
  };
  std::vector<Waypoint> waypoints;
  int reference_waypoint_id = 0;                         // :132
  double reference_waypoint_ratio[PP_NUM_LANES] = {0, 0, 0};  // :133

  Map() = default;
  ~Map() { pp_map_destroy(h_); }
  Map(const Map &) = delete;
  Map &operator=(const Map &) = delete;

  double get_lane_center_offset(int lane) const { return 4.0 * (lane + 0.5); }  // :84-88

  // :89-131.  The table is built by the library on the host (bit-identical to the
  // reference's Map::Init) and uploaded once.
  void Init(const std::vector<double> &map_waypoints_x, const std::vector<double> &map_waypoints_y) {
    pp_map_destroy(h_);
    h_ = nullptr;
    check(pp_map_create(map_waypoints_x.data(), map_waypoints_y.data(),
                        (int)map_waypoints_x.size(), &h_),
          "pp_map_create");
    fill_waypoints();
  }
  void InitFromCsv(const std::string &path) {  // the parsing of :1171-1191
    pp_map_destroy(h_);
    h_ = nullptr;
    check(pp_map_create_from_csv(path.c_str(), &h_), "pp_map_create_from_csv");
    fill_waypoints();
  }
  const pp_map *handle() const { return h_; }

  Waypoint &get_waypoint(int idx) {  // :134-137 (same unsigned arithmetic)
    return waypoints[(idx + waypoints.size()) % waypoints.size()];
  }
  double get_lane_length(int wp, int lane) { return lens_[wrap(wp) * PP_NUM_LANES + lane]; }  // :138-142

  // :143-197 — keeps the result on the object like the reference does
  void init_reference_waypoint(double x, double y) {
    ref_x_ = x;
    ref_y_ = y;
    detail::Dev<double> dx = detail::one(x), dy = detail::one(y), ratio(PP_NUM_LANES);
    detail::Dev<int32_t> wp(1);
    check(pp_init_reference_waypoint_batch(h_, dx.get(), dy.get(), wp.get(), ratio.get(), 1, nullptr),
          "pp_init_reference_waypoint_batch");
    reference_waypoint_id = wp.first();
    ratio.to_host(reference_waypoint_ratio);
  }

  // :199-275.  lane_mask is accepted for signature parity; the reference only ever passes
  // the default (all lanes).
  bool lane_matching(double x, double y, double &out_s, double &out_d, int &out_lane,
                     int *p_next_wp_id = nullptr, int lane_mask = 0xFFFF) {
    (void)lane_mask;
    double vs, vd;
    return match(x, y, 0, 0, out_s, out_d, out_lane, p_next_wp_id, vs, vd);
  }

  // :277-328
  Point get_lane_pos(double s, int lane, int &next_waypoint_id, double &next_waypoint_distance) {
    detail::Dev<double> rx = detail::one(ref_x_), ry = detail::one(ref_y_), ds = detail::one(s), ox(1),
                        oy(1), od(1);
    int32_t l = lane;
    detail::Dev<int32_t> dl(&l, 1), ow(1);
    check(pp_get_lane_pos_batch(h_, rx.get(), ry.get(), ds.get(), dl.get(), ox.get(), oy.get(),
                                ow.get(), od.get(), 1, nullptr),
          "pp_get_lane_pos_batch");
    next_waypoint_id = ow.first();
    next_waypoint_distance = od.first();
    return Point(ox.first(), oy.first());
  }

  // :330-358
  void project_speed(Point speed_vector, int next_wp_id, double *p_vs, double *p_vd) {
    int32_t wp = next_wp_id;
    detail::Dev<double> vx = detail::one(speed_vector.x), vy = detail::one(speed_vector.y), ovs(1),
                        ovd(1);
    detail::Dev<int32_t> dwp(&wp, 1);
    check(pp_project_speed_batch(h_, vx.get(), vy.get(), dwp.get(), ovs.get(), ovd.get(), 1, nullptr),
          "pp_project_speed_batch");
    *p_vs = ovs.first();
    *p_vd = ovd.first();
  }

  // the sensor-fusion loop body (:1336-1343) for one car: lane_matching + project_speed
  bool match_car(Car &c, int *p_next_wp_id = nullptr) {
    return match(c.x, c.y, c.vx, c.vy, c.s, c.d, c.lane, p_next_wp_id, c.vs, c.vd);
  }

 private:
  pp_map *h_ = nullptr;
  std::vector<double> lens_;
  double ref_x_ = 0, ref_y_ = 0;

  size_t wrap(int idx) const { return (idx + waypoints.size()) % waypoints.size(); }
  void fill_waypoints() {
    const int n = pp_map_num_waypoints(h_);
    std::vector<double> t((size_t)n * PP_MAP_STRIDE);
    check(pp_map_table(h_, t.data()), "pp_map_table");
    waypoints.resize(n);
    lens_.resize((size_t)n * PP_NUM_LANES);
    for (int i = 0; i < n; i++) {
      const double *r = &t[(size_t)i * PP_MAP_STRIDE];
      Waypoint &w = waypoints[i];
      w.ref = Point(r[0], r[1]);
      for (int l = 0; l < PP_NUM_LANES; l++) {
        w.lane_center[l] = Point(r[2 + 2 * l], r[3 + 2 * l]);
        lens_[(size_t)i * PP_NUM_LANES + l] = r[10 + l];
      }
      w.len = 0;
      w.nx = r[8];
      w.ny = r[9];
    }
  }
  bool match(double x, double y, double vx, double vy, double &s, double &d, int &lane,
             int *p_next_wp, double &vs, double &vd) {
    using detail::one;
    detail::Dev<double> rx = one(ref_x_), ry = one(ref_y_), dx = one(x), dy = one(y), dvx = one(vx),
                        dvy = one(vy), os(1), od(1), ovs(1), ovd(1);
    detail::Dev<int32_t> ok(1), ol(1), ow(1);
    check(pp_lane_matching_batch(h_, rx.get(), ry.get(), dx.get(), dy.get(), dvx.get(), dvy.get(),
                                 ok.get(), ol.get(), ow.get(), os.get(), od.get(), ovs.get(),
                                 ovd.get(), 1, nullptr),
          "pp_lane_matching_batch");
    if (!ok.first()) return false;  // the reference leaves the outputs untouched on failure
    s = os.first();
    d = od.first();
    lane = ol.first();
    vs = ovs.first();
    vd = ovd.first();
    if (p_next_wp) *p_next_wp = ow.first();
    return true;
  }
};

class LaneChangePlanner {  // src/main.cpp:361-485
 public:
  int calculate_target_lane(std::map<int, Car> &sensor_fusion_cars, int ego_lane, int target_lane,
                            double ego_s, double ego_vs, double delta_t0) {
    std::vector<int32_t> id, lane;
    std::vector<double> s, vs;
    for (auto &kv : sensor_fusion_cars) {
      id.push_back(kv.second.id);
      lane.push_back(kv.second.lane);
      s.push_back(kv.second.s);
      vs.push_back(kv.second.vs);
    }
    if (id.empty()) {  // keep the kernel's row length >= 1: one car that is "not in the map"
      id.push_back(0);
      lane.push_back(-1);
      s.push_back(0);
      vs.push_back(0);
    }
    const pp_config cfg = default_config();
    int32_t el = ego_lane, tl = target_lane;
    detail::Dev<int32_t> did(id), dlane(lane), del(&el, 1), dtl(&tl, 1), out(1);
    detail::Dev<double> ds(s), dvs(vs), des = detail::one(ego_s), devs = detail::one(ego_vs),
                        ddt = detail::one(delta_t0);
    check(pp_lane_change_batch(&cfg, did.get(), ds.get(), dvs.get(), dlane.get(), (int32_t)id.size(),
                               del.get(), dtl.get(), des.get(), devs.get(), ddt.get(), out.get(), 1,
                               nullptr),
          "pp_lane_change_batch");
    return out.first();
  }
};

class SpeedController {  // src/main.cpp:488-548
 public:
  double start_speed;
  double target_speed;
  double target_time;
  double time_shift;
  explicit SpeedController(double ego_speed)  // :493-501
      : start_speed(ego_speed), target_speed(0), target_time(0), time_shift(0) {
    run(3, 0, 0);
  }
  double get_speed(double current_t) { return run(0, current_t, 0); }                       // :503-512
  void add_limit_breakpoint(double new_target_speed, double new_target_time) {               // :513-533
    run(1, new_target_speed, new_target_time);
  }
  void override_speed(double current_t, double speed) { run(2, current_t, speed); }          // :534-547

 private:
  double run(int op, double a, double b) {
    using detail::one;
    detail::Dev<double> st = one(start_speed), tg = one(target_speed), tm = one(target_time),
                        sh = one(time_shift), da = one(a), db = one(b), out(1);
    check(pp_speed_controller_batch(op, st.get(), tg.get(), tm.get(), sh.get(), da.get(), db.get(),
                                    out.get(), 1, nullptr),
          "pp_speed_controller_batch");
    target_speed = tg.first();
    target_time = tm.first();
    time_shift = sh.first();
    return op == 0 ? out.first() : 0.0;
  }
};

class LimitSpeed {  // src/main.cpp:1052-1151
 public:
  double target_speed = 0;
  double target_time = 0;
  bool can_accelerate = true;
  uint32_t flags = 0;  // PP_F_COLLISION | BRAKE | MAXBRAKE | ADJUST | KEEP: the reference's prints

  void calculate(Car &follow_car, double next_s, double ego_s, double ego_speed, double ego_acc,
                 bool in_lane) {
    using detail::one;
    const pp_config cfg = default_config();
    int32_t il = in_lane ? 1 : 0;
    detail::Dev<double> vx = one(follow_car.vx), vy = one(follow_car.vy), ns = one(next_s),
                        es = one(ego_s), ev = one(ego_speed), ea = one(ego_acc), ls(1), lt(1), ss(1),
                        stt(1);
    detail::Dev<int32_t> dil(&il, 1);
    detail::Dev<uint32_t> fl(1);
    check(pp_limit_speed_batch(&cfg, vx.get(), vy.get(), ns.get(), es.get(), ev.get(), ea.get(),
                               dil.get(), ls.get(), lt.get(), ss.get(), stt.get(), fl.get(), 1,
                               nullptr),
          "pp_limit_speed_batch");
    target_speed = ls.first();
    target_time = lt.first();
    flags = fl.first();
    can_accelerate = !(flags & (PP_F_BRAKE | PP_F_MAXBRAKE));
  }
};

class TrajectoryBuilder {  // src/main.cpp:550-1049
 public:
  uint32_t flags = 0;  // PP_F_* raised while building (the reference prints them)

  // Same argument list as the reference.  ego_x/ego_y are what the glue passes: the last kept
  // previous point when prev_trajectory holds the 10 kept points, the telemetry pose otherwise.
  std::vector<Point> build(std::vector<Point> &prev_trajectory, double ego_x, double ego_y,
                           double ego_yaw, int ego_lane, int target_lane, double ego_d,
                           double ego_vd, Map &map, SpeedController &speed_controller) {
    (void)ego_lane;  // dead in the reference too (:611-636)
    using detail::one;
    const pp_config cfg = default_config();
    double px[PP_PREV_KEEP] = {0}, py[PP_PREV_KEEP] = {0};
    const int32_t pn = (int32_t)prev_trajectory.size();
    if (pn != 0 && pn != PP_PREV_KEEP)
      throw Error(PP_E_ARG, "TrajectoryBuilder::build: prev_trajectory must hold 0 or 10 points "
                            "(the glue keeps exactly 10, src/main.cpp:1261-1268)");
    for (int i = 0; i < pn; i++) {
      px[i] = prev_trajectory[i].x;
      py[i] = prev_trajectory[i].y;
    }
    int32_t tl = target_lane;
    detail::Dev<int32_t> dpn(&pn, 1), dtl(&tl, 1), on(1);
    detail::Dev<double> dpx(px, PP_PREV_KEEP), dpy(py, PP_PREV_KEEP), ex = one(ego_x), ey = one(ego_y),
                        yaw = one(ego_yaw), ed = one(ego_d), evd = one(ego_vd),
                        s0 = one(speed_controller.start_speed), s1 = one(speed_controller.target_speed),
                        s2 = one(speed_controller.target_time), ox(PP_PATH_LEN), oy(PP_PATH_LEN);
    detail::Dev<uint32_t> fl(1);
    check(pp_trajectory_build_batch(map.handle(), &cfg, dpn.get(), dpx.get(), dpy.get(), ex.get(),
                                    ey.get(), yaw.get(), dtl.get(), ed.get(), evd.get(), s0.get(),
                                    s1.get(), s2.get(), ox.get(), oy.get(), on.get(), fl.get(), 1,
                                    nullptr),
          "pp_trajectory_build_batch");
    flags = fl.first();
    const int n = on.first();
    const std::vector<double> x = ox.to_host(), y = oy.to_host();
    std::vector<Point> r(n);
    for (int i = 0; i < n; i++) r[i] = Point(x[i], y[i]);
    return r;
  }

  // The builder's control points alone (:638-768; a local of build() in the reference, which
  // writes them to trajectory.log as control_points=): (pos_x, pos_y) = the last kept previous
  // point, or the telemetry pose on a cold start; start_speed = the SpeedController's.
  static std::vector<Point> control_points(Map &map, double pos_x, double pos_y, int target_lane,
                                           double ego_d, double ego_vd, double start_speed) {
    using detail::one;
    int32_t tl = target_lane;
    detail::Dev<int32_t> dtl(&tl, 1), on(1);
    detail::Dev<double> px = one(pos_x), py = one(pos_y), ed = one(ego_d), evd = one(ego_vd),
                        s0 = one(start_speed), ox(6), oy(6);
    check(pp_control_points_batch(map.handle(), px.get(), py.get(), dtl.get(), ed.get(), evd.get(),
                                  s0.get(), ox.get(), oy.get(), on.get(), 1, nullptr),
          "pp_control_points_batch");
    const int n = on.first();
    const std::vector<double> x = ox.to_host(), y = oy.to_host();
    std::vector<Point> r(n);
    for (int i = 0; i < n; i++) r[i] = Point(x[i], y[i]);
    return r;
  }
};

namespace tk {
class spline {  // src/spline.h:284-396 (natural cubic through the points)
 public:
  void set_points(const std::vector<double> &x, const std::vector<double> &y) {
    if (x.size() != y.size() || x.size() < 3 || x.size() > 15)
      throw Error(PP_E_RANGE, "tk::spline::set_points: 3..15 knots");
    x_ = x;
    y_ = y;
  }
  double operator()(double q) const {
    detail::Dev<double> kx(x_), ky(y_), dq = detail::one(q), out(1);
    check(pp_spline_batch(kx.get(), ky.get(), (int32_t)x_.size(), dq.get(), 1, out.get(), 1, nullptr),
          "pp_spline_batch");
    return out.first();
  }

 private:
  std::vector<double> x_, y_;
};
}  // namespace tk

// ---- the planning step of onMessage, batched -------------------------------------
// One telemetry frame as the reference's lambda reads it (src/main.cpp:1233-1252,1297,1328-1334).
struct Frame {
  double car_x = 0, car_y = 0, car_yaw = 0, car_speed = 0;  // telemetry pose (deg, mph)
  std::vector<double> previous_path_x, previous_path_y;      // unconsumed points of the last plan
  int target_lane = 1;                                       // persistent planner state (:1195)
  std::vector<Car> sensor_fusion;                            // id, x, y, vx, vy
};
struct Plan {
  std::vector<double> next_x, next_y;  // what the reference sends back (:1450-1462)
  int target_lane = 1;                 // carry into the next frame
  int ego_lane = 0, ref_wp = 0;
  uint32_t flags = 0;
  double ego_s = 0, ego_d = 0, ego_vs = 0, ego_vd = 0, ego_speed = 0, ego_acc = 0;
  double target_speed = 0, target_time = 0;
  int next_car_id = -1, next_car_in_target_lane = -1;
  // the frame's sensor_fusion entries after the matching loop (:1325-1350): s, d, vs, vd, lane
  // filled in; lane == -1: lane matching failed, the reference erases the car (:1339)
  std::vector<Car> cars;
};

class Planner {
 public:
  explicit Planner(const Map &map) : map_(map), cfg_(default_config()) {}
  pp_config &config() { return cfg_; }

  // N frames -> N plans: marshals into the SoA layout of pp_frames and calls
  // pp_plan_batch_host_split (upload, the sm_100a pipeline, download).  The first PP_PREV_KEEP
  // points of a trajectory are the frame's own previous points (result_points =
  // prev_trajectory, src/main.cpp:578), so they are taken from the frame and only the new points
  // cross PCIe: the heads are aliased onto the previous-point arrays.
  std::vector<Plan> plan(const std::vector<Frame> &frames) {
    const size_t n = frames.size();
    size_t mc = 1;
    for (const Frame &f : frames) mc = f.sensor_fusion.size() > mc ? f.sensor_fusion.size() : mc;
    if (mc > PP_MAX_CARS) throw Error(PP_E_RANGE, "Planner::plan: more than PP_MAX_CARS cars in a frame");
    std::vector<double> ex(n), ey(n), eyaw(n), esp(n), px(n * PP_PREV_KEEP), py(n * PP_PREV_KEEP),
        cx(n * mc), cy(n * mc), cvx(n * mc), cvy(n * mc);
    std::vector<int32_t> pn(n), tl(n), nc(n), cid(n * mc);
    bool any_frozen = false;
    for (const Frame &f : frames)
      for (const Car &c : f.sensor_fusion) any_frozen = any_frozen || c.frozen;
    std::vector<int32_t> fz_lane(any_frozen ? n * mc : 0, -1);
    std::vector<double> fz_s(fz_lane.size()), fz_d(fz_lane.size()), fz_vs(fz_lane.size()),
        fz_vd(fz_lane.size());
    for (size_t i = 0; i < n; i++) {
      const Frame &f = frames[i];
      ex[i] = f.car_x;
      ey[i] = f.car_y;
      eyaw[i] = f.car_yaw;
      esp[i] = f.car_speed;
      pn[i] = (int32_t)f.previous_path_x.size();
      for (int k = 0; k < PP_PREV_KEEP && k < pn[i]; k++) {
        px[i * PP_PREV_KEEP + k] = f.previous_path_x[k];
        py[i * PP_PREV_KEEP + k] = f.previous_path_y[k];
      }
      tl[i] = f.target_lane;
      nc[i] = (int32_t)f.sensor_fusion.size();
      for (size_t j = 0; j < f.sensor_fusion.size(); j++) {
        const Car &c = f.sensor_fusion[j];
        cid[i * mc + j] = c.id;
        cx[i * mc + j] = c.x;
        cy[i * mc + j] = c.y;
        cvx[i * mc + j] = c.vx;
        cvy[i * mc + j] = c.vy;
        if (c.frozen) {
          fz_lane[i * mc + j] = c.lane;
          fz_s[i * mc + j] = c.s;
          fz_d[i * mc + j] = c.d;
          fz_vs[i * mc + j] = c.vs;
          fz_vd[i * mc + j] = c.vd;
        }
      }
    }
    pp_frames in;
    std::memset(&in, 0, sizeof in);
    if (any_frozen) {
      in.car_frozen_lane = fz_lane.data();
      in.car_frozen_s = fz_s.data();
      in.car_frozen_d = fz_d.data();
      in.car_frozen_vs = fz_vs.data();
      in.car_frozen_vd = fz_vd.data();
    }
    in.ego_x = ex.data();
    in.ego_y = ey.data();
    in.ego_yaw_deg = eyaw.data();
    in.ego_speed_mph = esp.data();
    in.prev_n = pn.data();
    in.prev_x = px.data();
    in.prev_y = py.data();
    in.target_lane_in = tl.data();
    in.n_cars = nc.data();
    in.car_id = cid.data();
    in.car_x = cx.data();
    in.car_y = cy.data();
    in.car_vx = cvx.data();
    in.car_vy = cvy.data();
    in.max_cars = (int32_t)mc;
    const size_t tail_len = PP_PATH_LEN - PP_PREV_KEEP;
    std::vector<double> tx(n * tail_len), ty(n * tail_len), d[8];
    for (auto &v : d) v.resize(n);
    std::vector<int32_t> np(n), el(n), rw(n), otl(n), id0(n), id1(n);
    std::vector<uint32_t> fl(n);
    pp_plans out;
    std::memset(&out, 0, sizeof out);
    out.n_points = np.data();
    out.ego_lane = el.data();
    out.ref_wp = rw.data();
    out.target_lane = otl.data();
    out.flags = fl.data();
    out.ego_s = d[0].data();
    out.ego_d = d[1].data();
    out.ego_vs = d[2].data();
    out.ego_vd = d[3].data();
    out.ego_speed = d[4].data();
    out.ego_acc = d[5].data();
    out.target_speed = d[6].data();
    out.target_time = d[7].data();
    out.next_car_id = id0.data();
    out.next_car_in_target_lane = id1.data();
    std::vector<double> cs(n * mc), cd(n * mc), cvs(n * mc), cvd(n * mc);
    std::vector<int32_t> cl(n * mc);
    out.car_s = cs.data();
    out.car_d = cd.data();
    out.car_vs = cvs.data();
    out.car_vd = cvd.data();
    out.car_lane = cl.data();
    pp_split_rows rows;
    rows.head_x = px.data();  // on return: the first points of every trajectory
    rows.head_y = py.data();
    rows.tail_x = tx.data();
    rows.tail_y = ty.data();
    check(pp_plan_batch_host_split(map_.handle(), &cfg_, &in, &out, &rows, (int64_t)n),
          "pp_plan_batch_host_split");
    std::vector<Plan> plans(n);
    for (size_t i = 0; i < n; i++) {
      Plan &p = plans[i];
      const size_t cnt = (size_t)np[i], head = cnt < (size_t)PP_PREV_KEEP ? cnt : (size_t)PP_PREV_KEEP;
      p.next_x.assign(px.begin() + i * PP_PREV_KEEP, px.begin() + i * PP_PREV_KEEP + head);
      p.next_y.assign(py.begin() + i * PP_PREV_KEEP, py.begin() + i * PP_PREV_KEEP + head);
      p.next_x.insert(p.next_x.end(), tx.begin() + i * tail_len, tx.begin() + i * tail_len + (cnt - head));
      p.next_y.insert(p.next_y.end(), ty.begin() + i * tail_len, ty.begin() + i * tail_len + (cnt - head));
      p.target_lane = otl[i];
      p.ego_lane = el[i];
      p.ref_wp = rw[i];
      p.flags = fl[i];
      p.ego_s = d[0][i];
      p.ego_d = d[1][i];
      p.ego_vs = d[2][i];
      p.ego_vd = d[3][i];
      p.ego_speed = d[4][i];
      p.ego_acc = d[5][i];
      p.target_speed = d[6][i];
      p.target_time = d[7][i];
      p.next_car_id = id0[i];
      p.next_car_in_target_lane = id1[i];
      p.cars = frames[i].sensor_fusion;
      for (size_t j = 0; j < p.cars.size(); j++) {
        Car &c = p.cars[j];
        c.s = cs[i * mc + j];
        c.d = cd[i * mc + j];
        c.vs = cvs[i * mc + j];
        c.vd = cvd[i * mc + j];
        c.lane = cl[i * mc + j];
      }
    }
    return plans;
  }
  Plan plan(const Frame &frame) { return plan(std::vector<Frame>(1, frame))[0]; }

  // The candidate sweep (pp_sweep_batch): 3 lanes x 16 target speeds x 8 target times through
  // SpeedController / TrajectoryBuilder, scored on the output points, best one returned.
  struct Swept {
    int best = -1;           // (lane * 16 + speed index) * 8 + time index
    double score = 0;
    std::vector<double> next_x, next_y;
    std::vector<double> scores;  // all PP_SWEEP_CANDS
    int lane() const { return best / (PP_SWEEP_SPEEDS * PP_SWEEP_TIMES); }
  };
  Swept sweep(const Frame &f) {
    const size_t mc = f.sensor_fusion.empty() ? 1 : f.sensor_fusion.size();
    if (mc > PP_MAX_CARS) throw Error(PP_E_RANGE, "Planner::sweep: more than PP_MAX_CARS cars");
    double px[PP_PREV_KEEP] = {0}, py[PP_PREV_KEEP] = {0};
    const int32_t pn = (int32_t)f.previous_path_x.size(), tl = f.target_lane,
                  nc = (int32_t)f.sensor_fusion.size();
    for (int k = 0; k < PP_PREV_KEEP && k < pn; k++) {
      px[k] = f.previous_path_x[k];
      py[k] = f.previous_path_y[k];
    }
    std::vector<int32_t> cid(mc, 0);
    std::vector<double> cx(mc, 0.0), cy(mc, 0.0), cvx(mc, 0.0), cvy(mc, 0.0);
    for (size_t j = 0; j < f.sensor_fusion.size(); j++) {
      cid[j] = f.sensor_fusion[j].id;
      cx[j] = f.sensor_fusion[j].x;
      cy[j] = f.sensor_fusion[j].y;
      cvx[j] = f.sensor_fusion[j].vx;
      cvy[j] = f.sensor_fusion[j].vy;
    }
    using detail::Dev;
    using detail::one;
    Dev<double> ex = one(f.car_x), ey = one(f.car_y), eyaw = one(f.car_yaw), esp = one(f.car_speed),
                dpx(px, PP_PREV_KEEP), dpy(py, PP_PREV_KEEP), dcx(cx), dcy(cy), dcvx(cvx), dcvy(cvy);
    Dev<int32_t> dpn(&pn, 1), dtl(&tl, 1), dnc(&nc, 1), dcid(cid);
    pp_frames in;
    std::memset(&in, 0, sizeof in);
    in.ego_x = ex.get();
    in.ego_y = ey.get();
    in.ego_yaw_deg = eyaw.get();
    in.ego_speed_mph = esp.get();
    in.prev_n = dpn.get();
    in.prev_x = dpx.get();
    in.prev_y = dpy.get();
    in.target_lane_in = dtl.get();
    in.n_cars = dnc.get();
    in.car_id = dcid.get();
    in.car_x = dcx.get();
    in.car_y = dcy.get();
    in.car_vx = dcvx.get();
    in.car_vy = dcvy.get();
    in.max_cars = (int32_t)mc;
    Dev<int32_t> best(1), npts(1);
    Dev<double> bs(1), nx(PP_PATH_LEN), ny(PP_PATH_LEN), sc(PP_SWEEP_CANDS);
    pp_sweep_out out;
    out.best = best.get();
    out.best_score = bs.get();
    out.next_x = nx.get();
    out.next_y = ny.get();
    out.n_points = npts.get();
    out.scores = sc.get();
    check(pp_sweep_batch(map_.handle(), &cfg_, &in, &out, 1, nullptr), "pp_sweep_batch");
    check(pp_dev_sync(), "pp_dev_sync");
    Swept r;
    r.best = best.first();
    r.score = bs.first();
    const int n = npts.first();
    const std::vector<double> x = nx.to_host(), y = ny.to_host();
    r.next_x.assign(x.begin(), x.begin() + n);
    r.next_y.assign(y.begin(), y.begin() + n);
    r.scores = sc.to_host();
    return r;
  }

 private:
  const Map &map_;
  pp_config cfg_;
};

// Closed-loop rollouts (pp_rollouts_*): n independent ego vehicles, each with its own synthetic
// traffic, stepped on the device against their own plans.
class Rollouts {
 public:
  Rollouts(const Map &map, int64_t n, int n_cars = 12, uint64_t seed = 0x5EED, int64_t first = 0)
      : n_(n), n_cars_(n_cars), cfg_(default_config()) {
    check(pp_rollouts_create(map.handle(), n, n_cars, seed, first, &h_), "pp_rollouts_create");
  }
  ~Rollouts() { pp_rollouts_destroy(h_); }
  Rollouts(const Rollouts &) = delete;
  Rollouts &operator=(const Rollouts &) = delete;
  void run(int64_t ticks, int consume_k = 1) {
    check(pp_rollouts_run(h_, &cfg_, ticks, consume_k, nullptr), "pp_rollouts_run");
    check(pp_dev_sync(), "pp_dev_sync");
  }
  struct Ego {
    std::vector<double> x, y, speed_mph;
    std::vector<int32_t> target_lane, path_n;
    int64_t tick = 0;
  };
  Ego ego() const {
    Ego e;
    e.x.resize(n_);
    e.y.resize(n_);
    e.speed_mph.resize(n_);
    e.target_lane.resize(n_);
    e.path_n.resize(n_);
    pp_rollout_state st;
    std::memset(&st, 0, sizeof st);
    st.ego_x = e.x.data();
    st.ego_y = e.y.data();
    st.ego_speed_mph = e.speed_mph.data();
    st.target_lane = e.target_lane.data();
    st.path_n = e.path_n.data();
    check(pp_rollouts_get_state(h_, &st), "pp_rollouts_get_state");
    e.tick = st.tick;
    return e;
  }
  // The incident monitor's record (pp.h, pp_rollout_incidents); count is [n][PP_INC_KINDS].
  struct Incidents {
    std::vector<int32_t> count, first_kind;
    std::vector<int64_t> first_tick;
    std::vector<double> distance_m, clean_m, best_clean_m, max_speed, max_acc, max_jerk;
  };
  Incidents incidents() const {
    Incidents r;
    r.count.resize((size_t)n_ * PP_INC_KINDS);
    r.first_kind.resize(n_);
    r.first_tick.resize(n_);
    for (auto *v : {&r.distance_m, &r.clean_m, &r.best_clean_m, &r.max_speed, &r.max_acc, &r.max_jerk})
      v->resize(n_);
    pp_rollout_incidents h;
    h.count = r.count.data();
    h.first_tick = r.first_tick.data();
    h.first_kind = r.first_kind.data();
    h.distance_m = r.distance_m.data();
    h.clean_m = r.clean_m.data();
    h.best_clean_m = r.best_clean_m.data();
    h.max_speed = r.max_speed.data();
    h.max_acc = r.max_acc.data();
    h.max_jerk = r.max_jerk.data();
    check(pp_rollouts_get_incidents(h_, &h), "pp_rollouts_get_incidents");
    return r;
  }
  // Traffic model (pp.h, PP_TRAFFIC_*), before the first tick only.
  void set_traffic(int model) { check(pp_rollouts_set_traffic(h_, model), "pp_rollouts_set_traffic"); }
  // The IDM traffic state (PP_TRAFFIC_IDM only); ego_s is [n][3].
  struct Traffic {
    std::vector<double> car_v0, car_acc, ego_s;
    std::vector<int32_t> ego_lanes;
  };
  Traffic traffic() const {
    Traffic t;
    t.car_v0.resize((size_t)n_ * n_cars_);
    t.car_acc.resize((size_t)n_ * n_cars_);
    t.ego_lanes.resize(n_);
    t.ego_s.resize((size_t)n_ * 3);
    pp_rollout_traffic h;
    h.car_v0 = t.car_v0.data();
    h.car_acc = t.car_acc.data();
    h.ego_lanes = t.ego_lanes.data();
    h.ego_s = t.ego_s.data();
    check(pp_rollouts_get_traffic(h_, &h), "pp_rollouts_get_traffic");
    return t;
  }
  // Flight recorder (pp.h, pp_rollouts_set_recorder), before the first tick only.
  void set_recorder(int window, uint32_t triggers) {
    check(pp_rollouts_set_recorder(h_, window, triggers), "pp_rollouts_set_recorder");
    window_ = window;
  }
  // The recorded windows of `rows` (all rollouts when empty): m rows of window() slots, oldest
  // first; the frame fields are in pp_frames layout with max_cars = n_cars (frame (i, j) at
  // i * window() + j).
  struct Recording {
    std::vector<int64_t> trigger_tick, tick;
    std::vector<uint32_t> trigger_bits;
    std::vector<int32_t> consume_k, prev_n, target_lane_in, n_cars, car_id;
    std::vector<double> ego_x, ego_y, ego_yaw_deg, ego_speed_mph, prev_x, prev_y, car_x, car_y,
        car_vx, car_vy;
  };
  Recording recording(const std::vector<int64_t> &rows = std::vector<int64_t>()) const {
    const size_t m = rows.empty() ? (size_t)n_ : rows.size(), mw = m * (size_t)window_,
                 mwc = mw * (size_t)n_cars_;
    Recording o;
    o.trigger_tick.resize(m);
    o.trigger_bits.resize(m);
    o.tick.resize(mw);
    for (auto *v : {&o.consume_k, &o.prev_n, &o.target_lane_in, &o.n_cars}) v->resize(mw);
    for (auto *v : {&o.ego_x, &o.ego_y, &o.ego_yaw_deg, &o.ego_speed_mph}) v->resize(mw);
    o.prev_x.resize(mw * PP_PREV_KEEP);
    o.prev_y.resize(mw * PP_PREV_KEEP);
    for (auto *v : {&o.car_x, &o.car_y, &o.car_vx, &o.car_vy}) v->resize(mwc);
    o.car_id.resize(mwc);
    pp_rollout_recording h;
    h.trigger_tick = o.trigger_tick.data();
    h.trigger_bits = o.trigger_bits.data();
    h.tick = o.tick.data();
    h.consume_k = o.consume_k.data();
    h.ego_x = o.ego_x.data();
    h.ego_y = o.ego_y.data();
    h.ego_yaw_deg = o.ego_yaw_deg.data();
    h.ego_speed_mph = o.ego_speed_mph.data();
    h.prev_x = o.prev_x.data();
    h.prev_y = o.prev_y.data();
    h.car_x = o.car_x.data();
    h.car_y = o.car_y.data();
    h.car_vx = o.car_vx.data();
    h.car_vy = o.car_vy.data();
    h.prev_n = o.prev_n.data();
    h.target_lane_in = o.target_lane_in.data();
    h.n_cars = o.n_cars.data();
    h.car_id = o.car_id.data();
    check(pp_rollouts_get_recording(h_, rows.empty() ? nullptr : rows.data(), (int64_t)m, &h),
          "pp_rollouts_get_recording");
    return o;
  }
  // Near-miss measures (pp.h, pp_rollouts_set_surrogate), before the first tick only.
  void set_surrogate(bool on = true) {
    check(pp_rollouts_set_surrogate(h_, on ? 1 : 0), "pp_rollouts_set_surrogate");
  }
  // The near-miss record; time_hist is [n][PP_SSM_MEASURES][PP_SSM_BINS].
  struct Surrogate {
    std::vector<double> min_ttc_front, min_ttc_rear, min_thw;
    std::vector<int64_t> min_ttc_front_tick;
    std::vector<int32_t> time_hist;
  };
  Surrogate surrogate() const {
    Surrogate o;
    for (auto *v : {&o.min_ttc_front, &o.min_ttc_rear, &o.min_thw}) v->resize(n_);
    o.min_ttc_front_tick.resize(n_);
    o.time_hist.resize((size_t)n_ * PP_SSM_MEASURES * PP_SSM_BINS);
    pp_rollout_surrogate h;
    h.min_ttc_front = o.min_ttc_front.data();
    h.min_ttc_rear = o.min_ttc_rear.data();
    h.min_thw = o.min_thw.data();
    h.min_ttc_front_tick = o.min_ttc_front_tick.data();
    h.time_hist = o.time_hist.data();
    check(pp_rollouts_get_surrogate(h_, &h), "pp_rollouts_get_surrogate");
    return o;
  }
  // The totals (pp.h, pp_rollouts_surrogate_totals), copied to the host.
  std::vector<int64_t> surrogate_totals() const {
    detail::Dev<int64_t> dev(PP_SSM_TOTALS_LEN);
    check(pp_rollouts_surrogate_totals(h_, dev.get(), nullptr), "pp_rollouts_surrogate_totals");
    check(pp_dev_sync(), "pp_dev_sync");
    return dev.to_host();
  }
  // Episode restarts (pp.h, pp_rollouts_set_restart), before the first tick only; 0 = off.
  void set_restart(uint32_t triggers) {
    check(pp_rollouts_set_restart(h_, triggers), "pp_rollouts_set_restart");
  }
  // The restart record; by_bit is [n][PP_INC_KINDS + 1].
  struct Restarts {
    std::vector<int64_t> episodes, by_bit, episode_tick, ended_lap;
    std::vector<double> episode_m, ended_m;
  };
  Restarts restarts() const {
    Restarts o;
    for (auto *v : {&o.episodes, &o.episode_tick, &o.ended_lap}) v->resize(n_);
    o.by_bit.resize((size_t)n_ * (PP_INC_KINDS + 1));
    o.episode_m.resize(n_);
    o.ended_m.resize(n_);
    pp_rollout_restarts h;
    h.episodes = o.episodes.data();
    h.by_bit = o.by_bit.data();
    h.episode_tick = o.episode_tick.data();
    h.episode_m = o.episode_m.data();
    h.ended_m = o.ended_m.data();
    h.ended_lap = o.ended_lap.data();
    check(pp_rollouts_get_restarts(h_, &h), "pp_rollouts_get_restarts");
    return o;
  }
  // The totals (pp.h, pp_rollouts_restart_totals), copied to the host.
  std::vector<int64_t> restart_totals() const {
    detail::Dev<int64_t> dev(PP_RST_TOTALS_LEN);
    check(pp_rollouts_restart_totals(h_, dev.get(), nullptr), "pp_rollouts_restart_totals");
    check(pp_dev_sync(), "pp_dev_sync");
    return dev.to_host();
  }

 private:
  pp_rollouts *h_ = nullptr;
  int64_t n_;
  int n_cars_;
  int window_ = 0;
  pp_config cfg_;
};

}  // namespace pp

#endif  // PP_B200_HPP
