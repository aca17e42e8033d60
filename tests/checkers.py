"""Test-side bindings of the two CPU checkers under oracle/ (TEST INFRASTRUCTURE).

  Checker("ref")    oracle/_ref/libppref.so  — the reference's own sources, compiled
  Checker("oracle") oracle/libpporacle.so    — the plain-C restatement

Both export the same C functions with the prefixes ppref_ / ppo_.
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / reference
arm may import this module.
"""
from __future__ import annotations

import ctypes as C
import importlib.util
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG_DIR = os.path.join(ROOT, "carnd-path-planning-project_b200")
MAP_CSV = os.path.join(ROOT, "data", "highway_map.csv")


def load_pkg():
    """Import the product package (its directory name has hyphens)."""
    name = "carnd_path_planning_project_b200"
    if name in sys.modules:
        return sys.modules[name]
    spec = importlib.util.spec_from_file_location(
        name, os.path.join(PKG_DIR, "__init__.py"), submodule_search_locations=[PKG_DIR])
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def load_abi():
    name = "carnd_path_planning_project_b200.abi"
    if name in sys.modules:
        return sys.modules[name]
    spec = importlib.util.spec_from_file_location(name, os.path.join(PKG_DIR, "abi.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


abi = load_abi()

_PATHS = {
    "ref": (os.path.join(ROOT, "oracle", "_ref", "libppref.so"), "ppref_"),
    # the same sources with the reference's own flags (no -O): a CPU-baseline figure only
    "ref_O0": (os.path.join(ROOT, "oracle", "_ref", "libppref_O0.so"), "ppref_"),
    "oracle": (os.path.join(ROOT, "oracle", "libpporacle.so"), "ppo_"),
}


def available(kind: str) -> bool:
    return os.path.exists(_PATHS[kind][0])


def _p(a):
    return C.c_void_p(a.ctypes.data)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _cfg_fields(cfg):
    return tuple(getattr(cfg, name) for name, _ in abi.Config._fields_ if name != "reserved")


# Planner tunables the parity tests run besides the reference's literals:
#   tight  every field moved; speed overrides, curvature adjustments, KEEP / ADJUST common
#   loose  fast and hard-accelerating: ego speeds of 30-40 m/s in the rollouts
#   max25  an integral max_speed, for the (int)max_speed truncation of the lane statistics
#   edges  a relaxed_acc whose significand is all ones (no cached reciprocal shortcut), zero
#          leeway and safety distance, a weak braking deceleration
CONFIGS = {
    "default": {},
    "tight": dict(relaxed_acc=3.0, min_relaxed_acc_while_braking=2.5, maximum_acc=4.0,
                  max_speed=17.5, car_length=5.5, safety_distance=4.0, keep_distance=25.0,
                  keep_distance_leeway=3.0, test_fast_lane_change=1),
    "loose": dict(relaxed_acc=30.0, maximum_acc=30.0, max_speed=40.0),
    "max25": dict(max_speed=25.0),
    "edges": dict(relaxed_acc=3.9999999999999996, min_relaxed_acc_while_braking=0.5,
                  keep_distance_leeway=0.0, safety_distance=0.0),
}


def config(name: str = "default", **fields):
    """abi.Config: the named entry of CONFIGS over the defaults, then `fields` over that."""
    cfg = abi.default_config()
    for k, v in {**CONFIGS[name], **fields}.items():
        assert hasattr(cfg, k), k
        setattr(cfg, k, v)
    return cfg


def hold_over(fb, plans, rng, frac=0.3, stale=True):
    """Turn about `frac` of the matched car slots of `fb` (plans: a plan of fb with per-car
    outputs) into cars held over from an earlier message (pp_frames::car_frozen_*): their
    car_x / car_y become NaN, so only the frozen values can place them.  stale=False freezes a
    slot at exactly its own matched values; stale=True moves s by up to 30 m, d by up to 1.5 m
    (the lane follows d) and scales vs by 0.5-1.5.  Returns (frames, mask of frozen slots)."""
    out = fb.slice(0, fb.n).add_frozen()
    live = np.arange(fb.max_cars)[None, :] < fb.n_cars[:, None]
    pick = live & (plans.car_lane >= 0) & (rng.random(live.shape) < frac)
    k = int(pick.sum())
    s, d, vs, vd = (getattr(plans, n)[pick] for n in ("car_s", "car_d", "car_vs", "car_vd"))
    lane = plans.car_lane[pick]
    if stale:
        s = s + rng.uniform(-30.0, 30.0, k)
        d = np.clip(d + rng.uniform(-1.5, 1.5, k), 0.1, 11.9)
        lane = np.clip(np.floor(d / 4.0), 0, 2).astype(np.int32)
        vs = vs * rng.uniform(0.5, 1.5, k)
    out.car_frozen_lane[pick] = lane
    out.car_frozen_s[pick], out.car_frozen_d[pick] = s, d
    out.car_frozen_vs[pick], out.car_frozen_vd[pick] = vs, vd
    out.car_x[pick] = np.nan
    out.car_y[pick] = np.nan
    return out, pick


class Checker:
    def __init__(self, kind: str, map_csv: str = MAP_CSV):
        path, self.pre = _PATHS[kind]
        if not os.path.exists(path):
            raise FileNotFoundError(f"{path} not built (run `make -C oracle`)")
        self.kind = kind
        self.lib = C.CDLL(path)
        fn = self._fn("map_create_from_csv")
        fn.restype = C.c_void_p
        self.map = C.c_void_p(fn(map_csv.encode()))
        if not self.map.value:
            raise RuntimeError("map load failed")
        self._fn("map_num_waypoints").restype = C.c_int
        self.n_wp = self._fn("map_num_waypoints")(self.map)
        self._fn("observable_flags").restype = C.c_uint32
        self.observable_flags = self._fn("observable_flags")()

    def _fn(self, name):
        return getattr(self.lib, self.pre + name)

    def _cfg_call(self, name, cfg):
        """(function, leading config argument) for a planning function: the oracle's _cfg entry
        point with any config; the reference's own code knows only its literals."""
        if cfg is None:
            return self._fn(name), ()
        if self.kind != "oracle":
            if _cfg_fields(cfg) != _cfg_fields(abi.default_config()):
                raise ValueError(f"checker {self.kind!r} plans with the default config only")
            return self._fn(name), ()
        return self._fn(name + "_cfg"), (C.byref(cfg),)

    def map_from_points(self, wx, wy):
        fn = self._fn("map_create")
        fn.restype = C.c_void_p
        wx, wy = _f64(wx), _f64(wy)
        self.map = C.c_void_p(fn(_p(wx), _p(wy), C.c_int(len(wx))))
        self.n_wp = len(wx)

    def map_table(self):
        out = np.zeros((self.n_wp, abi.MAP_STRIDE))
        self._fn("map_table")(self.map, _p(out))
        return out

    def plan(self, frames, threads: int = 1, want_flags: bool = True, diag=True, cars=True,
             cfg=None):
        plans = abi.PlanBatch(frames.n, frames.max_cars, diag=diag, cars=cars)
        self.plan_into(frames, plans, threads, want_flags, cfg)
        return plans

    def plan_with_log(self, frames, log_path: str):
        """ref only: plan with the reference's trajectory.log sites writing to log_path."""
        assert self.kind.startswith("ref")
        plans = abi.PlanBatch(frames.n, frames.max_cars, diag=True, cars=True)
        fs, ps = frames.struct(), plans.struct()
        rc = self.lib.ppref_plan_frames_log(self.map, C.byref(fs), C.byref(ps), C.c_int64(frames.n),
                                            log_path.encode())
        assert rc == 0, rc
        return plans

    def plan_into(self, frames, plans, threads: int = 1, want_flags: bool = False, cfg=None):
        fs, ps = frames.struct(), plans.struct()
        fn, pre = self._cfg_call("plan_frames", cfg)
        rc = fn(self.map, *pre, C.byref(fs), C.byref(ps), C.c_int64(frames.n), C.c_int(threads),
                C.c_int(1 if want_flags else 0))
        assert rc == 0, rc

    # ---- unit functions ----
    def distancesq_pt_seg(self, px, py, ax, ay, bx, by):
        args = [_f64(a) for a in (px, py, ax, ay, bx, by)]
        n = len(args[0])
        outs = [np.zeros(n) for _ in range(4)]
        self._fn("distancesq_pt_seg")(*[_p(a) for a in args], *[_p(o) for o in outs],
                                      C.c_int64(n))
        return outs  # d2, rnom, rdenom, snom

    def init_reference_waypoint(self, x, y):
        x, y = _f64(x), _f64(y)
        n = len(x)
        wp = np.zeros(n, np.int32)
        ratio = np.zeros((n, 3))
        self._fn("init_reference_waypoint")(self.map, _p(x), _p(y), _p(wp), _p(ratio),
                                            C.c_int64(n))
        return wp, ratio

    def lane_matching(self, rx, ry, x, y, vx, vy):
        a = [_f64(v) for v in (rx, ry, x, y, vx, vy)]
        n = len(a[0])
        ok, lane, nwp = (np.zeros(n, np.int32) for _ in range(3))
        s, d, vs, vd = (np.zeros(n) for _ in range(4))
        self._fn("lane_matching")(self.map, *[_p(v) for v in a], _p(ok), _p(lane), _p(nwp),
                                  _p(s), _p(d), _p(vs), _p(vd), C.c_int64(n))
        return dict(ok=ok, lane=lane, next_wp=nwp, s=s, d=d, vs=vs, vd=vd)

    def get_lane_pos(self, rx, ry, s, lane):
        rx, ry, s = _f64(rx), _f64(ry), _f64(s)
        lane = _i32(lane)
        n = len(rx)
        ox, oy, od = np.zeros(n), np.zeros(n), np.zeros(n)
        owp = np.zeros(n, np.int32)
        self._fn("get_lane_pos")(self.map, _p(rx), _p(ry), _p(s), _p(lane), _p(ox), _p(oy),
                                 _p(owp), _p(od), C.c_int64(n))
        return ox, oy, owp, od

    def spline(self, kx, ky, q):
        kx, ky, q = _f64(kx), _f64(ky), _f64(q)
        ns, nk = kx.shape
        nq = q.shape[1]
        out = np.zeros((ns, nq))
        self._fn("spline")(_p(kx), _p(ky), C.c_int32(nk), _p(q), C.c_int32(nq), _p(out),
                           C.c_int64(ns))
        return out

    def closest_waypoint(self, x, y, mx, my):
        x, y, mx, my = map(_f64, (x, y, mx, my))
        out = np.zeros(len(x), np.int32)
        self._fn("closest_waypoint")(_p(x), _p(y), _p(mx), _p(my), C.c_int32(len(mx)), _p(out),
                                     C.c_int64(len(x)))
        return out

    def next_waypoint(self, x, y, th, mx, my):
        x, y, th, mx, my = map(_f64, (x, y, th, mx, my))
        out = np.zeros(len(x), np.int32)
        self._fn("next_waypoint")(_p(x), _p(y), _p(th), _p(mx), _p(my), C.c_int32(len(mx)),
                                  _p(out), C.c_int64(len(x)))
        return out

    def get_frenet(self, x, y, th, mx, my):
        x, y, th, mx, my = map(_f64, (x, y, th, mx, my))
        os_, od = np.zeros(len(x)), np.zeros(len(x))
        self._fn("get_frenet")(_p(x), _p(y), _p(th), _p(mx), _p(my), C.c_int32(len(mx)),
                               _p(os_), _p(od), C.c_int64(len(x)))
        return os_, od

    def get_xy(self, s, d, ms, mx, my):
        s, d, ms, mx, my = map(_f64, (s, d, ms, mx, my))
        ox, oy = np.zeros(len(s)), np.zeros(len(s))
        self._fn("get_xy")(_p(s), _p(d), _p(ms), _p(mx), _p(my), C.c_int32(len(mx)), _p(ox),
                           _p(oy), C.c_int64(len(s)))
        return ox, oy

    def lane_change(self, car_id, car_s, car_vs, car_lane, ego_lane, target_lane, ego_s, ego_vs,
                    dt0, cfg=None):
        car_id, car_lane = _i32(car_id), _i32(car_lane)
        car_s, car_vs = _f64(car_s), _f64(car_vs)
        ego_lane, target_lane = _i32(ego_lane), _i32(target_lane)
        ego_s, ego_vs, dt0 = _f64(ego_s), _f64(ego_vs), _f64(dt0)
        n, nc = car_id.shape
        out = np.zeros(n, np.int32)
        fn, pre = self._cfg_call("lane_change", cfg)
        fn(*pre, _p(car_id), _p(car_s), _p(car_vs), _p(car_lane), C.c_int32(nc), _p(ego_lane),
           _p(target_lane), _p(ego_s), _p(ego_vs), _p(dt0), _p(out), C.c_int64(n))
        return out

    def limit_speed(self, car_vx, car_vy, next_s, ego_s, ego_speed, ego_acc, in_lane, cfg=None):
        a = [_f64(v) for v in (car_vx, car_vy, next_s, ego_s, ego_speed, ego_acc)]
        in_lane = _i32(in_lane)
        n = len(in_lane)
        outs = [np.zeros(n) for _ in range(4)]
        flags = np.zeros(n, np.uint32)
        fn, pre = self._cfg_call("limit_speed", cfg)
        fn(*pre, *[_p(v) for v in a], _p(in_lane), *[_p(o) for o in outs], _p(flags),
           C.c_int64(n))
        return dict(ls_speed=outs[0], ls_time=outs[1], sc_speed=outs[2], sc_time=outs[3],
                    flags=flags)

    def trajectory_build(self, prev_n, prev_x, prev_y, ego_x, ego_y, yaw, target_lane, ego_d,
                         ego_vd, sc_start, sc_target, sc_time, cfg=None):
        prev_n, target_lane = _i32(prev_n), _i32(target_lane)
        f = [_f64(v) for v in (prev_x, prev_y, ego_x, ego_y, yaw)]
        g = [_f64(v) for v in (ego_d, ego_vd, sc_start, sc_target, sc_time)]
        n = len(prev_n)
        ox = np.full((n, abi.PATH_LEN), np.nan)
        oy = np.full((n, abi.PATH_LEN), np.nan)
        on = np.zeros(n, np.int32)
        fl = np.zeros(n, np.uint32)
        fn, pre = self._cfg_call("trajectory_build", cfg)
        fn(self.map, *pre, _p(prev_n), *[_p(v) for v in f], _p(target_lane), *[_p(v) for v in g],
           _p(ox), _p(oy), _p(on), _p(fl), C.c_int64(n))
        return ox, oy, on, fl

    # ---- simulator model of the closed-loop rollouts (oracle only) ----
    def sim_frames(self, state, n_cars):
        """frame <- state.  `state`: the package's RolloutStateHost."""
        assert self.kind == "oracle"
        fb = abi.FrameBatch(state.n, max(n_cars, 1))
        st, fs = state.struct(), fb.struct()
        self._fn("sim_frames")(self.map, C.byref(st), C.c_int64(state.n), C.c_int32(n_cars),
                               C.byref(fs))
        return fb

    def sim_advance(self, state, n_cars, seed, first, consume_k, plans):
        """state <- simulator step(plan), in place (tick incremented)."""
        assert self.kind == "oracle"
        st, ps = state.struct(), plans.struct()
        self._fn("sim_advance")(self.map, C.byref(st), C.c_int64(state.n), C.c_int32(n_cars),
                                C.c_uint64(seed), C.c_int64(first), C.c_int32(consume_k),
                                C.byref(ps))
        state.tick = int(st.tick)

    def lambda_sequence(self, frames):
        """ref only: the untouched onMessage lambda over a frame SEQUENCE."""
        assert self.kind == "ref"
        ox = np.full((frames.n, abi.PATH_LEN), np.nan)
        oy = np.full((frames.n, abi.PATH_LEN), np.nan)
        on = np.zeros(frames.n, np.int32)
        fs = frames.struct()
        cwd = os.path.join(ROOT, "oracle")  # ../data/highway_map.csv resolves from here
        rc = self.lib.ppref_lambda_sequence(cwd.encode(), C.byref(fs), C.c_int64(frames.n),
                                            _p(ox), _p(oy), _p(on))
        assert rc == 0, rc
        return ox, oy, on
