"""B200-native batched highway path planner — Python binding of the C ABI.

The product is ``libpp_b200.so`` (hand-written sm_100a CUDA kernels behind the
``extern "C"`` entry points of ``include/pp.h``).  This module is a thin ctypes
wrapper used by the tests and ``bench.py``; PyTorch appears only as the owner of
device memory / streams and for ``torch.distributed`` plumbing.

There is no CPU planning path here: if the shared library is missing the import
fails, and if no CUDA device is usable every planning call raises ``PPError``.
"""
from __future__ import annotations

import ctypes as C
import os

# more hardware work queues than the default 8 (see pp_api.cu: the planner uses nine streams);
# read at CUDA context creation, so set it before anything touches the device
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

import numpy as np

from . import abi
from .abi import (Config, FrameBatch, Frames, PlanBatch, Plans, default_config, FLAG, FLAG_NAMES,
                  NUM_FLAGS, STATS_LEN, PATH_LEN, PREV_KEEP, MAP_STRIDE, FSTATS_LEN, FSTAT_NMIN,
                  FSTAT_NAMES, COMM_ID_BYTES)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpp_b200.so")
ROOT = os.path.dirname(_HERE)
MAP_CSV = os.path.join(ROOT, "data", "highway_map.csv")

# every symbol include/pp.h declares (tests check the library exports them all)
EXPORTS = [
    "pp_version", "pp_init", "pp_strerror", "pp_last_cuda_error", "pp_device_count", "pp_config_default",
    "pp_map_create", "pp_map_create_from_csv", "pp_map_destroy", "pp_map_num_waypoints",
    "pp_map_table", "pp_plan_batch", "pp_plan_batch_host", "pp_plan_batch_host_split", "pp_stats_batch",
    "pp_set_kernel_variant", "pp_launch_count", "pp_distancesq_pt_seg_batch",
    "pp_init_reference_waypoint_batch", "pp_lane_matching_batch", "pp_get_lane_pos_batch",
    "pp_spline_batch", "pp_closest_waypoint_batch", "pp_next_waypoint_batch",
    "pp_get_frenet_batch", "pp_get_xy_batch", "pp_synth_frames", "pp_selftest_math",
    "pp_lane_change_batch", "pp_limit_speed_batch", "pp_trajectory_build_batch",
    "pp_set_phase_timing", "pp_get_phase_ms", "pp_speed_controller_batch",
    "pp_project_speed_batch", "pp_control_points_batch",
    "pp_dev_alloc", "pp_dev_free", "pp_host_alloc", "pp_host_free", "pp_dev_upload", "pp_dev_download", "pp_dev_sync",
    "pp_dev_set", "pp_stream_create", "pp_stream_sync", "pp_stream_destroy",
    "pp_rollouts_create", "pp_rollouts_destroy", "pp_rollouts_run", "pp_rollouts_last",
    "pp_rollouts_get_state", "pp_rollouts_stats", "pp_rollouts_set_lean", "pp_rollouts_set_groups",
    "pp_rollouts_get_incidents", "pp_rollouts_incident_totals", "pp_rollouts_set_traffic",
    "pp_rollouts_get_traffic", "pp_rollouts_set_recorder", "pp_rollouts_get_recording",
    "pp_rollouts_set_surrogate", "pp_rollouts_get_surrogate", "pp_rollouts_surrogate_totals",
    "pp_sweep_batch",
    "pp_set_pipes", "pp_plan_stats_batch", "pp_synth_frames_dev", "pp_fstats_batch",
    "pp_comm_unique_id", "pp_comm_init_rank", "pp_comm_init_all", "pp_comm_destroy",
    "pp_comm_group_begin", "pp_comm_group_end", "pp_stats_reduce",
]


class PPError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python {os.path.join(_HERE, 'build.py')}` "
            "(there is no fallback implementation)")
    lib = C.CDLL(LIB_PATH)
    lib.pp_strerror.restype = C.c_char_p
    lib.pp_last_cuda_error.restype = C.c_char_p
    lib.pp_launch_count.restype = C.c_int64
    return lib


lib = _load()


def _check(rc: int, what: str):
    if rc != 0:
        msg = lib.pp_strerror(rc).decode()
        detail = lib.pp_last_cuda_error().decode() if rc == -2 else ""
        raise PPError(f"{what} failed: {msg} {detail}".strip())


def launch_count() -> int:
    return int(lib.pp_launch_count())


def device_count() -> int:
    return int(lib.pp_device_count())


def set_kernel_variant(v: int):
    _check(lib.pp_set_kernel_variant(C.c_int(v)), "pp_set_kernel_variant")


def set_pipes(n: int):
    _check(lib.pp_set_pipes(C.c_int(n)), "pp_set_pipes")


def set_phase_timing(on: bool):
    _check(lib.pp_set_phase_timing(C.c_int(1 if on else 0)), "pp_set_phase_timing")


def get_phase_ms():
    """(ms[5] = prep, cars, decide, emit, slow summed over the chunks since the last call, chunks)."""
    ms = (C.c_double * 5)()
    chunks = C.c_int64(0)
    _check(lib.pp_get_phase_ms(ms, C.byref(chunks)), "pp_get_phase_ms")
    return [float(v) for v in ms], int(chunks.value)


def _ptr(t):
    """Raw address of a torch tensor / numpy array / None."""
    if t is None:
        return None
    if isinstance(t, np.ndarray):
        return t.ctypes.data
    return t.data_ptr()


class Map:
    """Owner of a pp_map (host table + device copy on the current CUDA device)."""

    def __init__(self, csv_path: str = MAP_CSV, points=None):
        self._h = C.c_void_p()
        if points is not None:
            wx = np.ascontiguousarray(points[0], dtype=np.float64)
            wy = np.ascontiguousarray(points[1], dtype=np.float64)
            rc = lib.pp_map_create(C.c_void_p(wx.ctypes.data), C.c_void_p(wy.ctypes.data),
                                   C.c_int(len(wx)), C.byref(self._h))
        else:
            rc = lib.pp_map_create_from_csv(csv_path.encode(), C.byref(self._h))
        _check(rc, "pp_map_create")
        self.n = int(lib.pp_map_num_waypoints(self._h))

    @property
    def handle(self):
        return self._h

    def table(self) -> np.ndarray:
        out = np.zeros((self.n, MAP_STRIDE))
        _check(lib.pp_map_table(self._h, C.c_void_p(out.ctypes.data)), "pp_map_table")
        return out

    def close(self):
        if self._h:
            lib.pp_map_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def synth_frames(m: Map, n: int, n_cars: int = 12, seed: int = 0x5EED, first_frame: int = 0,
                 rare_permille: int = 20, max_cars: int | None = None,
                 out: FrameBatch | None = None) -> FrameBatch:
    """SURVEY §8d synthetic workload (host generator inside the library)."""
    fb = out if out is not None else FrameBatch(n, max_cars if max_cars is not None else n_cars)
    s = fb.struct()
    _check(lib.pp_synth_frames(m.handle, C.c_uint64(seed), C.c_int64(first_frame), C.c_int64(n),
                               C.c_int32(n_cars), C.c_int32(rare_permille), C.byref(s)),
           "pp_synth_frames")
    return fb


def plan_batch_host(m: Map, frames: FrameBatch, plans: PlanBatch | None = None,
                    cfg: Config | None = None, diag: bool = True, cars: bool = True) -> PlanBatch:
    """pp_plan_batch_host: host buffers in, host buffers out (copies inside)."""
    cfg = cfg or default_config()
    plans = plans or PlanBatch(frames.n, frames.max_cars, diag=diag, cars=cars)
    fs, ps = frames.struct(), plans.struct()
    _check(lib.pp_plan_batch_host(m.handle, C.byref(cfg), C.byref(fs), C.byref(ps),
                                  C.c_int64(frames.n)), "pp_plan_batch_host")
    return plans


class _Pinned:
    """Owner of one pp_host_alloc block."""

    def __init__(self, nbytes: int):
        self.p = C.c_void_p()
        _check(lib.pp_host_alloc(C.byref(self.p), C.c_size_t(nbytes)), "pp_host_alloc")

    def __del__(self):
        try:
            if self.p:
                lib.pp_host_free(self.p)
                self.p = C.c_void_p()
        except Exception:
            pass


def pinned_empty(shape, dtype=np.float64) -> np.ndarray:
    """numpy array in page-locked host memory (pp_host_alloc); freed with its last view."""
    dt = np.dtype(dtype)
    shape = (shape,) if np.isscalar(shape) else tuple(shape)
    nbytes = int(np.prod(shape, dtype=np.int64)) * dt.itemsize
    owner = _Pinned(max(nbytes, 1))
    buf = (C.c_char * max(nbytes, 1)).from_address(owner.p.value)
    buf._owner = owner  # the array's base keeps the block alive
    return np.frombuffer(buf, dtype=dt, count=int(np.prod(shape, dtype=np.int64))).reshape(shape)


def pinned_like(a: np.ndarray) -> np.ndarray:
    out = pinned_empty(a.shape, a.dtype)
    out[...] = a
    return out


def plan_batch_host_split(m: Map, frames: FrameBatch, plans: PlanBatch, head_x, head_y, tail_x,
                          tail_y, cfg: Config | None = None) -> PlanBatch:
    """pp_plan_batch_host_split: as plan_batch_host, but the trajectories come back as
    head[n][PREV_KEEP] (written only for frames that kept no previous points; may be the
    frames' own prev_x / prev_y arrays) and tail[n][PATH_LEN - PREV_KEEP]; `plans` must have
    next_x = next_y = None."""
    cfg = cfg or default_config()
    fs, ps = frames.struct(), plans.struct()
    rows = abi.SplitRows(_ptr(head_x), _ptr(head_y), _ptr(tail_x), _ptr(tail_y))
    _check(lib.pp_plan_batch_host_split(m.handle, C.byref(cfg), C.byref(fs), C.byref(ps),
                                        C.byref(rows), C.c_int64(frames.n)),
           "pp_plan_batch_host_split")
    return plans


class DeviceFrames:
    """Frames resident in HBM (torch tensors), layout of pp_frames."""

    def __init__(self, frames: FrameBatch, device="cuda"):
        import torch
        self.n, self.max_cars = frames.n, frames.max_cars
        self.t = {k: torch.from_numpy(v).to(device) for k, v in frames.arrays().items()}
        if getattr(frames, "car_frozen_lane", None) is not None:  # optional held-over cars
            for name, _ in abi.FROZEN_FIELDS:
                self.t[name] = torch.from_numpy(getattr(frames, name)).to(device)

    @classmethod
    def empty(cls, n: int, max_cars: int, device="cuda") -> "DeviceFrames":
        import torch
        self = cls.__new__(cls)
        self.n, self.max_cars = n, max_cars
        tmap = {np.float64: torch.float64, np.int32: torch.int32}
        self.t = {name: torch.empty((n,) + abi._inner(kind, max_cars), dtype=tmap[dt], device=device)
                  for name, dt, kind in abi.FRAME_FIELDS}
        return self

    def to_host(self) -> FrameBatch:
        fb = FrameBatch(self.n, self.max_cars)
        for k, v in self.t.items():
            setattr(fb, k, v.cpu().numpy())
        return fb

    def struct(self) -> Frames:
        s = Frames()
        for k, v in self.t.items():
            setattr(s, k, v.data_ptr())
        s.max_cars = self.max_cars
        return s

    def nbytes(self) -> int:
        return sum(v.numel() * v.element_size() for v in self.t.values())


class DevicePlans:
    """Plans resident in HBM (torch tensors), layout of pp_plans."""

    def __init__(self, n: int, max_cars: int, device="cuda", diag: bool = True, cars: bool = False):
        import torch
        self.n, self.max_cars = n, max_cars
        fields = list(abi.PLAN_CORE) + (abi.PLAN_DIAG if diag else []) + \
            (abi.PLAN_CARS if cars else [])
        tmap = {np.float64: torch.float64, np.int32: torch.int32, np.uint32: torch.int32}
        self.t = {}
        for name, dt, kind in abi.PLAN_FIELDS:
            if name in fields:
                shape = (n,) + abi._inner(kind, max_cars)
                self.t[name] = torch.zeros(shape, dtype=tmap[dt], device=device)

    def struct(self) -> Plans:
        s = Plans()
        for name, _, _ in abi.PLAN_FIELDS:
            setattr(s, name, self.t[name].data_ptr() if name in self.t else None)
        return s

    def to_host(self) -> PlanBatch:
        pb = PlanBatch(self.n, self.max_cars, diag="ego_s" in self.t, cars="car_s" in self.t)
        for name, dt, _ in abi.PLAN_FIELDS:
            if name in self.t:
                a = self.t[name].cpu().numpy()
                setattr(pb, name, a.view(np.uint32) if dt == np.uint32 else a)
        return pb

    def nbytes(self) -> int:
        return sum(v.numel() * v.element_size() for v in self.t.values())


def plan_batch(m: Map, frames: DeviceFrames, plans: DevicePlans, cfg: Config | None = None,
               stream=None, n: int | None = None):
    """pp_plan_batch on device-resident buffers; asynchronous on `stream`
    (an int cudaStream_t, default: torch's current stream)."""
    import torch
    cfg = cfg or default_config()
    if stream is None:
        stream = torch.cuda.current_stream().cuda_stream
    fs, ps = frames.struct(), plans.struct()
    _check(lib.pp_plan_batch(m.handle, C.byref(cfg), C.byref(fs), C.byref(ps),
                             C.c_int64(frames.n if n is None else n), C.c_void_p(stream)),
           "pp_plan_batch")


def plan_stats_batch(m: Map, frames: DeviceFrames, plans: DevicePlans, cfg: Config | None = None,
                     stream=None, out=None):
    """pp_plan_stats_batch: plan and aggregate in one call -> int64[STATS_LEN] device tensor."""
    import torch
    cfg = cfg or default_config()
    if stream is None:
        stream = torch.cuda.current_stream().cuda_stream
    if out is None:
        out = torch.empty(STATS_LEN, dtype=torch.int64, device=next(iter(plans.t.values())).device)
    fs, ps = frames.struct(), plans.struct()
    _check(lib.pp_plan_stats_batch(m.handle, C.byref(cfg), C.byref(fs), C.byref(ps),
                                   C.c_int64(frames.n), C.c_void_p(out.data_ptr()),
                                   C.c_void_p(stream)), "pp_plan_stats_batch")
    return out


def stats_batch(plans: DevicePlans, stream=None):
    """pp_stats_batch -> int64[STATS_LEN] torch tensor on the device."""
    import torch
    if stream is None:
        stream = torch.cuda.current_stream().cuda_stream
    out = torch.zeros(STATS_LEN, dtype=torch.int64, device=next(iter(plans.t.values())).device)
    ps = plans.struct()
    _check(lib.pp_stats_batch(C.byref(ps), C.c_int64(plans.n), C.c_void_p(out.data_ptr()),
                              C.c_void_p(stream)), "pp_stats_batch")
    return out


def fstats_batch(plans: DevicePlans, stream=None, out=None):
    """pp_fstats_batch -> float64[FSTATS_LEN] torch tensor on the device (minima, then maxima)."""
    import torch
    if stream is None:
        stream = torch.cuda.current_stream().cuda_stream
    if out is None:
        out = torch.empty(FSTATS_LEN, dtype=torch.float64, device=next(iter(plans.t.values())).device)
    ps = plans.struct()
    _check(lib.pp_fstats_batch(C.byref(ps), C.c_int64(plans.n), C.c_void_p(out.data_ptr()),
                               C.c_void_p(stream)), "pp_fstats_batch")
    return out


def synth_frames_dev(m: Map, n: int, n_cars: int = 12, seed: int = 0x5EED, first_frame: int = 0,
                     rare_permille: int = 20, max_cars: int | None = None,
                     out: "DeviceFrames | None" = None, stream=None) -> "DeviceFrames":
    """pp_synth_frames_dev: the synthetic workload generated in HBM (same bits as synth_frames)."""
    import torch
    if stream is None:
        stream = torch.cuda.current_stream().cuda_stream
    if out is None:
        out = DeviceFrames.empty(n, max_cars if max_cars is not None else max(n_cars, 1))
    s = out.struct()
    _check(lib.pp_synth_frames_dev(m.handle, C.c_uint64(seed), C.c_int64(first_frame), C.c_int64(n),
                                   C.c_int32(n_cars), C.c_int32(rare_permille), C.byref(s),
                                   C.c_void_p(stream)), "pp_synth_frames_dev")
    return out


class Comm:
    """An ncclComm_t made through the C ABI (pp_comm_*): one process per GPU.  `exchange` ships
    rank 0's 128-byte id to the other ranks (bytes -> bytes; e.g. a torch.distributed broadcast);
    world == 1 needs none."""

    def __init__(self, rank: int = 0, world: int = 1, exchange=None):
        self.rank, self.world = rank, world
        ident = (C.c_ubyte * COMM_ID_BYTES)()
        if rank == 0:
            _check(lib.pp_comm_unique_id(ident), "pp_comm_unique_id")
        if world > 1:
            raw = exchange(bytes(ident))
            ident = (C.c_ubyte * COMM_ID_BYTES).from_buffer_copy(raw)
        self._h = C.c_void_p()
        _check(lib.pp_comm_init_rank(ident, C.c_int(rank), C.c_int(world), C.byref(self._h)),
               "pp_comm_init_rank")

    def stats_reduce(self, stats=None, fstats=None, stream=None):
        """pp_stats_reduce: in-place ncclSum of int64 `stats`, ncclMin / ncclMax of f64 `fstats`."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
        _check(lib.pp_stats_reduce(self._h, C.c_void_p(_ptr(stats)), C.c_void_p(_ptr(fstats)),
                                   C.c_void_p(stream)), "pp_stats_reduce")

    def close(self):
        if self._h:
            lib.pp_comm_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class RolloutStateHost:
    """Host copy of the simulator state of a Rollouts object (numpy arrays)."""

    def __init__(self, n: int, n_cars: int):
        self.n, self.n_cars, self.tick = n, n_cars, 0
        for name, dt, kind in abi.ROLLOUT_STATE_FIELDS:
            inner = {0: (), "path": (abi.PATH_LEN,), "cars": (n_cars,)}[kind]
            setattr(self, name, np.zeros((n,) + inner, dtype=dt))

    def struct(self) -> abi.RolloutState:
        s = abi.RolloutState()
        for name, _, _ in abi.ROLLOUT_STATE_FIELDS:
            setattr(s, name, getattr(self, name).ctypes.data)
        s.tick = self.tick
        return s


class Rollouts:
    """Closed-loop rollouts (BASELINE config 3): pp_rollouts_* of include/pp.h."""

    def __init__(self, m: Map, n: int, n_cars: int = 12, seed: int = 0x5EED, first: int = 0,
                 lean: bool = False):
        self.map, self.n, self.n_cars = m, n, n_cars
        self._h = C.c_void_p()
        _check(lib.pp_rollouts_create(m.handle, C.c_int64(n), C.c_int32(n_cars), C.c_uint64(seed),
                                      C.c_int64(first), C.byref(self._h)), "pp_rollouts_create")
        if lean:
            _check(lib.pp_rollouts_set_lean(self._h, C.c_int(1)), "pp_rollouts_set_lean")

    def set_groups(self, groups: int):
        """Stream groups per tick (0 = automatic)."""
        _check(lib.pp_rollouts_set_groups(self._h, C.c_int(groups)), "pp_rollouts_set_groups")

    def run(self, ticks: int, consume_k: int = 1, cfg: Config | None = None, stream=None):
        import torch
        cfg = cfg or default_config()
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
        _check(lib.pp_rollouts_run(self._h, C.byref(cfg), C.c_int64(ticks), C.c_int32(consume_k),
                                   C.c_void_p(stream)), "pp_rollouts_run")

    def state(self) -> RolloutStateHost:
        st = RolloutStateHost(self.n, self.n_cars)
        s = st.struct()
        _check(lib.pp_rollouts_get_state(self._h, C.byref(s)), "pp_rollouts_get_state")
        st.tick = int(s.tick)
        return st

    def last(self):
        """(FrameBatch, PlanBatch) of the last tick, copied to the host."""
        import torch
        fs, ps = Frames(), Plans()
        _check(lib.pp_rollouts_last(self._h, C.byref(fs), C.byref(ps)), "pp_rollouts_last")
        torch.cuda.synchronize()
        mc = max(self.n_cars, 1)
        fb = FrameBatch(self.n, mc)
        for name, arr in fb.arrays().items():
            _check(lib.pp_dev_download(C.c_void_p(arr.ctypes.data), C.c_void_p(getattr(fs, name)),
                                       C.c_size_t(arr.nbytes)), "pp_dev_download")
        pb = PlanBatch(self.n, mc, diag=True, cars=True)
        for name, _, _ in abi.PLAN_FIELDS:
            arr = getattr(pb, name)
            if getattr(ps, name):  # lean rollouts leave the diagnostics out
                _check(lib.pp_dev_download(C.c_void_p(arr.ctypes.data), C.c_void_p(getattr(ps, name)),
                                           C.c_size_t(arr.nbytes)), "pp_dev_download")
        return fb, pb

    def stats(self, stream=None):
        import torch
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
        out = torch.zeros(STATS_LEN, dtype=torch.int64, device="cuda")
        _check(lib.pp_rollouts_stats(self._h, C.c_void_p(out.data_ptr()), C.c_void_p(stream)),
               "pp_rollouts_stats")
        return out

    def incidents(self) -> dict:
        """The incident monitor's record (include/pp.h, pp_rollout_incidents) as numpy arrays:
        count [n][INC_KINDS] (columns in the order of abi.INC_NAMES), first_tick / first_kind [n]
        (-1: none), distance_m, clean_m, best_clean_m, max_speed, max_acc, max_jerk [n]."""
        out = {name: np.zeros((self.n, abi.INC_KINDS) if kind else (self.n,), dtype=dt)
               for name, dt, kind in abi.INC_FIELDS}
        s = abi.RolloutIncidents(*[a.ctypes.data for a in out.values()])
        _check(lib.pp_rollouts_get_incidents(self._h, C.byref(s)), "pp_rollouts_get_incidents")
        return out

    def set_traffic(self, model):
        """Select the traffic model before the first tick: abi.TRAFFIC_CONSTANT (default) or
        abi.TRAFFIC_IDM (car following, include/pp.h), or their names "constant" / "idm"."""
        if isinstance(model, str):
            model = abi.TRAFFIC_MODELS[model]
        _check(lib.pp_rollouts_set_traffic(self._h, C.c_int(model)), "pp_rollouts_set_traffic")

    def traffic(self) -> dict:
        """The IDM traffic state (only under abi.TRAFFIC_IDM) as numpy arrays: car_v0, car_acc
        [n][n_cars], and the ego's lane state the next tick reads, ego_lanes [n] (bit L: the ego
        leads lane L) and ego_s [n][3]."""
        inner = {"cars": (self.n_cars,), 0: (), "lanes": (3,)}
        out = {name: np.zeros((self.n,) + inner[kind], dtype=dt)
               for name, dt, kind in abi.TRAFFIC_FIELDS}
        s = abi.RolloutTraffic(*[a.ctypes.data for a in out.values()])
        _check(lib.pp_rollouts_get_traffic(self._h, C.byref(s)), "pp_rollouts_get_traffic")
        return out

    def set_recorder(self, window: int, triggers=0):
        """Switch the flight recorder on before the first tick (include/pp.h): keep each rollout's
        frames of its last `window` ticks (0 = off) and freeze them at the first tick in which a
        trigger fires.  `triggers` is a bit mask or an iterable of names of abi.REC_NAMES (the
        incident kinds of abi.INC_NAMES and "nonfinite")."""
        mask = abi.rec_mask(triggers)
        if not 0 <= mask < 1 << 32 or not -2**31 <= window < 2**31:
            raise PPError(f"pp_rollouts_set_recorder failed: window {window} / mask {mask:#x}")
        _check(lib.pp_rollouts_set_recorder(self._h, C.c_int32(window), C.c_uint32(mask)),
               "pp_rollouts_set_recorder")
        self.rec_window = int(window)

    def recorder_triggers(self) -> dict:
        """trigger_tick (int64, -1: not frozen) and trigger_bits (uint32) of every rollout."""
        out = {"trigger_tick": np.zeros(self.n, np.int64), "trigger_bits": np.zeros(self.n, np.uint32)}
        s = abi.RolloutRecording(trigger_tick=out["trigger_tick"].ctypes.data,
                                 trigger_bits=out["trigger_bits"].ctypes.data)
        _check(lib.pp_rollouts_get_recording(self._h, None, C.c_int64(self.n), C.byref(s)),
               "pp_rollouts_get_recording")
        return out

    def recording(self, rollouts=None) -> dict:
        """The recorded windows of `rollouts` (indices; None: all) -> dict: trigger_tick,
        trigger_bits [m], tick, consume_k [m][W] (oldest first; tick -1: slot not filled) and
        "frames", a FrameBatch of m * W frames (frame (i, j) at i * W + j; unfilled slots are all
        0), ready for the device planner or the CPU oracle."""
        rows = None if rollouts is None else np.ascontiguousarray(rollouts, dtype=np.int64).reshape(-1)
        m = self.n if rows is None else len(rows)
        w = getattr(self, "rec_window", 0)
        fb = FrameBatch(m * w, max(self.n_cars, 1))
        out = {"trigger_tick": np.zeros(m, np.int64), "trigger_bits": np.zeros(m, np.uint32),
               "tick": np.zeros((m, w), np.int64), "consume_k": np.zeros((m, w), np.int32)}
        s = abi.RolloutRecording()
        for name, _, kind in abi.REC_FIELDS:
            a = out[name] if kind != "frame" else getattr(fb, name)
            setattr(s, name, a.ctypes.data if a.size else None)
        # a raw address must cross as c_void_p: a bare int is passed as a 32-bit C int
        _check(lib.pp_rollouts_get_recording(self._h, None if rows is None else C.c_void_p(rows.ctypes.data),
                                             C.c_int64(m), C.byref(s)), "pp_rollouts_get_recording")
        out["frames"] = fb
        return out

    def set_surrogate(self, on: bool = True):
        """Switch the near-miss measures on (or off) before the first tick (include/pp.h): time to
        collision ahead and behind, time headway, their minima and exposure histograms."""
        _check(lib.pp_rollouts_set_surrogate(self._h, C.c_int(1 if on else 0)),
               "pp_rollouts_set_surrogate")

    def surrogate(self) -> dict:
        """The near-miss record (include/pp.h, pp_rollout_surrogate) as numpy arrays:
        min_ttc_front, min_ttc_rear, min_thw [n] (s, inf: never defined), min_ttc_front_tick [n]
        (-1: never), time_hist [n][SSM_MEASURES][SSM_BINS] (ticks' weights in units of 0.02 s;
        measures in the order of abi.SSM_NAMES, bins below abi.SSM_EDGES)."""
        inner = {0: (), "hist": (abi.SSM_MEASURES, abi.SSM_BINS)}
        out = {name: np.zeros((self.n,) + inner[kind], dtype=dt) for name, dt, kind in abi.SSM_FIELDS}
        s = abi.RolloutSurrogate(*[a.ctypes.data for a in out.values()])
        _check(lib.pp_rollouts_get_surrogate(self._h, C.byref(s)), "pp_rollouts_get_surrogate")
        return out

    def surrogate_totals(self, stream=None):
        """pp_rollouts_surrogate_totals -> int64[SSM_TOTALS_LEN] device tensor: time_hist summed
        over the rollouts (entry m * SSM_BINS + b), then the rollouts per bin of their minima
        (entry SSM_TOTAL_MIN + m * SSM_BINS + b)."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
        out = torch.empty(abi.SSM_TOTALS_LEN, dtype=torch.int64, device="cuda")
        _check(lib.pp_rollouts_surrogate_totals(self._h, C.c_void_p(out.data_ptr()),
                                                C.c_void_p(stream)), "pp_rollouts_surrogate_totals")
        return out

    def incident_totals(self, stream=None):
        """pp_rollouts_incident_totals -> int64[INC_TOTALS_LEN] device tensor: counts per kind,
        rollouts with at least one incident, driven millimetres."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
        out = torch.empty(abi.INC_TOTALS_LEN, dtype=torch.int64, device="cuda")
        _check(lib.pp_rollouts_incident_totals(self._h, C.c_void_p(out.data_ptr()),
                                               C.c_void_p(stream)), "pp_rollouts_incident_totals")
        return out

    def close(self):
        if self._h:
            lib.pp_rollouts_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def sweep_batch(m: Map, frames: DeviceFrames, cfg: Config | None = None, want_scores: bool = True,
                stream=None):
    """pp_sweep_batch (BASELINE config 4) on device-resident frames -> dict of torch tensors:
    best [N] int32, best_score [N], next_x/next_y [N][50], n_points [N], scores [N][384]."""
    import torch
    cfg = cfg or default_config()
    if stream is None:
        stream = torch.cuda.current_stream().cuda_stream
    n = frames.n
    out = {"best": torch.zeros(n, dtype=torch.int32, device="cuda"),
           "best_score": torch.zeros(n, dtype=torch.float64, device="cuda"),
           "next_x": torch.zeros((n, abi.PATH_LEN), dtype=torch.float64, device="cuda"),
           "next_y": torch.zeros((n, abi.PATH_LEN), dtype=torch.float64, device="cuda"),
           "n_points": torch.zeros(n, dtype=torch.int32, device="cuda"),
           "scores": torch.zeros((n, abi.SWEEP_CANDS), dtype=torch.float64, device="cuda")
           if want_scores else None}
    so = abi.SweepOut()
    for k, v in out.items():
        setattr(so, k, v.data_ptr() if v is not None else None)
    fs = frames.struct()
    _check(lib.pp_sweep_batch(m.handle, C.byref(cfg), C.byref(fs), C.byref(so), C.c_int64(n),
                              C.c_void_p(stream)), "pp_sweep_batch")
    return out
