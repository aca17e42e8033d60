"""ctypes mirror of include/pp.h plus host-side (numpy) frame / plan containers.

This module only describes memory layouts; it contains no planning code.  The
same structs are handed to libpp_b200.so (the product) and, by the tests, to
the CPU checkers the tests own.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

NUM_LANES = 3
PREV_KEEP = 10
PATH_LEN = 50
MAX_CARS = 64
MAP_STRIDE = 13

OK = 0

FLAG_NAMES = [
    "EGO_MATCH_FAIL", "CAR_DROPPED", "COLLISION", "BRAKE", "MAXBRAKE", "ADJUST", "KEEP",
    "SPLINE_INPUT_ERR", "FALLBACK", "ACC_OVERRIDE", "CURV_ADJUST", "LANE_SWITCH_NEG", "VETO",
    "ACCT_HIGH", "ACCN_HIGH", "SPLINE_WARNING", "CLOSED_RANGE", "CLOSED_AHEAD", "CLOSED_BEHIND",
    "TRANSFORM_ERR", "COLD_START",
]
NUM_FLAGS = len(FLAG_NAMES)
FLAG = {name: 1 << i for i, name in enumerate(FLAG_NAMES)}

STAT_FRAMES = 0
STAT_POINTS = 1
STAT_TARGET_LANE0 = 2
STAT_EGO_LANE0 = 5
STAT_LANE_CHANGES = 8
STAT_FLAG0 = 9
STAT_XSUM = STAT_FLAG0 + NUM_FLAGS
STATS_LEN = STAT_XSUM + 1

# f64 min / max statistics (pp_fstats_batch): entries [0, FSTAT_NMIN) are minima
FSTAT_NAMES = ["min_ego_speed", "min_target_speed", "min_step_speed", "max_ego_speed",
               "max_target_speed", "max_step_speed", "max_acc"]
FSTAT_NMIN = 3
FSTATS_LEN = len(FSTAT_NAMES)
COMM_ID_BYTES = 128

_dp = C.c_void_p  # every array pointer crosses the ABI as a raw address


class Config(C.Structure):
    _fields_ = [
        ("relaxed_acc", C.c_double),
        ("min_relaxed_acc_while_braking", C.c_double),
        ("maximum_acc", C.c_double),
        ("max_speed", C.c_double),
        ("car_length", C.c_double),
        ("safety_distance", C.c_double),
        ("keep_distance", C.c_double),
        ("keep_distance_leeway", C.c_double),
        ("test_fast_lane_change", C.c_int32),
        ("reserved", C.c_int32),
    ]


FRAME_FIELDS = [  # (name, dtype, inner) ; inner: 0 scalar, 'prev', 'cars'
    ("ego_x", np.float64, 0),
    ("ego_y", np.float64, 0),
    ("ego_yaw_deg", np.float64, 0),
    ("ego_speed_mph", np.float64, 0),
    ("prev_n", np.int32, 0),
    ("prev_x", np.float64, "prev"),
    ("prev_y", np.float64, "prev"),
    ("target_lane_in", np.int32, 0),
    ("n_cars", np.int32, 0),
    ("car_id", np.int32, "cars"),
    ("car_x", np.float64, "cars"),
    ("car_y", np.float64, "cars"),
    ("car_vx", np.float64, "cars"),
    ("car_vy", np.float64, "cars"),
]

PLAN_FIELDS = [  # inner: 0 scalar, 'path', 'cars'
    ("next_x", np.float64, "path"),
    ("next_y", np.float64, "path"),
    ("n_points", np.int32, 0),
    ("ego_lane", np.int32, 0),
    ("ref_wp", np.int32, 0),
    ("target_lane", np.int32, 0),
    ("flags", np.uint32, 0),
    ("ego_s", np.float64, 0),
    ("ego_d", np.float64, 0),
    ("ego_vs", np.float64, 0),
    ("ego_vd", np.float64, 0),
    ("ego_speed", np.float64, 0),
    ("ego_acc", np.float64, 0),
    ("target_speed", np.float64, 0),
    ("target_time", np.float64, 0),
    ("next_car_id", np.int32, 0),
    ("next_car_in_target_lane", np.int32, 0),
    ("car_s", np.float64, "cars"),
    ("car_d", np.float64, "cars"),
    ("car_vs", np.float64, "cars"),
    ("car_vd", np.float64, "cars"),
    ("car_lane", np.int32, "cars"),
    ("car_next_wp", np.int32, "cars"),
]
PLAN_CORE = ["next_x", "next_y", "n_points", "ego_lane", "ref_wp", "target_lane", "flags"]
PLAN_DIAG = ["ego_s", "ego_d", "ego_vs", "ego_vd", "ego_speed", "ego_acc", "target_speed",
             "target_time", "next_car_id", "next_car_in_target_lane"]
PLAN_CARS = ["car_s", "car_d", "car_vs", "car_vd", "car_lane", "car_next_wp"]


# optional inputs (NULL unless set): cars held over from earlier messages (pp.h, pp_frames)
FROZEN_FIELDS = [("car_frozen_lane", np.int32), ("car_frozen_s", np.float64),
                 ("car_frozen_d", np.float64), ("car_frozen_vs", np.float64),
                 ("car_frozen_vd", np.float64)]


class Frames(C.Structure):
    _fields_ = [(n, _dp) for n, _, _ in FRAME_FIELDS] + [("max_cars", C.c_int32),
                                                         ("reserved", C.c_int32)] + \
               [(n, _dp) for n, _ in FROZEN_FIELDS]


class Plans(C.Structure):
    _fields_ = [(n, _dp) for n, _, _ in PLAN_FIELDS]


class SplitRows(C.Structure):
    """pp_split_rows (pp_plan_batch_host_split): [n][PREV_KEEP] heads, [n][PATH_LEN - PREV_KEEP] tails."""
    _fields_ = [(n, _dp) for n in ("head_x", "head_y", "tail_x", "tail_y")]


SWEEP_LANES, SWEEP_SPEEDS, SWEEP_TIMES = 3, 16, 8
SWEEP_CANDS = SWEEP_LANES * SWEEP_SPEEDS * SWEEP_TIMES
SWEEP_BAD = 1e9


class SweepOut(C.Structure):
    _fields_ = [(n, _dp) for n in ("best", "best_score", "next_x", "next_y", "n_points", "scores")]


ROLLOUT_STATE_FIELDS = [  # (name, dtype, inner) ; inner: 0 scalar, 'path', 'cars'
    ("ego_x", np.float64, 0), ("ego_y", np.float64, 0), ("ego_yaw_deg", np.float64, 0),
    ("ego_speed_mph", np.float64, 0), ("path_n", np.int32, 0), ("path_x", np.float64, "path"),
    ("path_y", np.float64, "path"), ("target_lane", np.int32, 0), ("car_lane", np.int32, "cars"),
    ("car_wp", np.int32, "cars"), ("car_ratio", np.float64, "cars"),
    ("car_speed", np.float64, "cars"),
]


class RolloutState(C.Structure):
    _fields_ = [(n, _dp) for n, _, _ in ROLLOUT_STATE_FIELDS] + [("tick", C.c_int64)]


# incident monitor of the rollouts (pp_rollout_incidents): kinds in the order of PP_INC_*
INC_NAMES = ["collision_front", "collision_rear", "over_speed", "over_acc", "over_jerk",
             "out_of_lane", "off_road"]
INC = {name: i for i, name in enumerate(INC_NAMES)}
INC_KINDS = len(INC_NAMES)
INC_TOTAL_ROLLOUTS = INC_KINDS      # pp_rollouts_incident_totals: rollouts with an incident
INC_TOTAL_MM = INC_KINDS + 1        # ... driven distance in millimetres
INC_TOTALS_LEN = INC_KINDS + 2
INC_HISTORY = 70                   # driven points the jerk reaches back (PP_INC_HISTORY)
INC_FIELDS = [  # (name, dtype, inner) ; inner: 0 scalar, 'kinds'
    ("count", np.int32, "kinds"), ("first_tick", np.int64, 0), ("first_kind", np.int32, 0),
    ("distance_m", np.float64, 0), ("clean_m", np.float64, 0), ("best_clean_m", np.float64, 0),
    ("max_speed", np.float64, 0), ("max_acc", np.float64, 0), ("max_jerk", np.float64, 0),
]


class RolloutIncidents(C.Structure):
    _fields_ = [(n, _dp) for n, _, _ in INC_FIELDS]


# traffic models of the rollouts (pp_rollouts_set_traffic) and the IDM parameters (PP_TRF_*)
TRAFFIC_CONSTANT = 0
TRAFFIC_IDM = 1
TRAFFIC_MODELS = {"constant": TRAFFIC_CONSTANT, "idm": TRAFFIC_IDM}
TRF_ACC = 1.5
TRF_DEC = 3.0
TRF_MAX_DEC = 9.0
TRF_HEADWAY = 1.2
TRF_MIN_GAP = 2.0
TRF_GAP_FLOOR = 0.1
TRF_EGO_CORRIDOR = 3.0
TRAFFIC_FIELDS = [  # (name, dtype, inner) ; inner: 'cars', 0 scalar, 'lanes'
    ("car_v0", np.float64, "cars"), ("car_acc", np.float64, "cars"),
    ("ego_lanes", np.int32, 0), ("ego_s", np.float64, "lanes"),
]


class RolloutTraffic(C.Structure):
    _fields_ = [(n, _dp) for n, _, _ in TRAFFIC_FIELDS]


# flight recorder of the rollouts (pp_rollouts_set_recorder): trigger bits are the PP_INC_* kinds
# plus REC_NONFINITE (distance_m not finite)
REC_NONFINITE = INC_KINDS
REC_NAMES = INC_NAMES + ["nonfinite"]
REC_MAX_WINDOW = 1024
REC_FIELDS = [  # (name, dtype, inner) ; inner: 0 per row, 'window' per slot, else a frame field
    ("trigger_tick", np.int64, 0), ("trigger_bits", np.uint32, 0),
    ("tick", np.int64, "window"), ("consume_k", np.int32, "window"),
    ("ego_x", np.float64, "frame"), ("ego_y", np.float64, "frame"),
    ("ego_yaw_deg", np.float64, "frame"), ("ego_speed_mph", np.float64, "frame"),
    ("prev_x", np.float64, "frame"), ("prev_y", np.float64, "frame"),
    ("car_x", np.float64, "frame"), ("car_y", np.float64, "frame"),
    ("car_vx", np.float64, "frame"), ("car_vy", np.float64, "frame"),
    ("prev_n", np.int32, "frame"), ("target_lane_in", np.int32, "frame"),
    ("n_cars", np.int32, "frame"), ("car_id", np.int32, "frame"),
]


class RolloutRecording(C.Structure):
    _fields_ = [(n, _dp) for n, _, _ in REC_FIELDS]


# near-miss measures of the rollouts (pp_rollouts_set_surrogate), in the order of PP_SSM_*
SSM_NAMES = ["ttc_front", "ttc_rear", "thw"]
SSM = {name: i for i, name in enumerate(SSM_NAMES)}
SSM_MEASURES = len(SSM_NAMES)
SSM_EDGES = [0.5, 1.0, 1.5, 2.0, 3.0, 4.0, 6.0, 8.0]  # s, upper bin edges (PP_SSM_EDGES)
SSM_BINS = len(SSM_EDGES)
SSM_TOTAL_MIN = SSM_MEASURES * SSM_BINS  # pp_rollouts_surrogate_totals: rollouts per bin of the minima
SSM_TOTALS_LEN = 2 * SSM_MEASURES * SSM_BINS
SSM_FIELDS = [  # (name, dtype, inner) ; inner: 0 scalar, 'hist' [SSM_MEASURES][SSM_BINS]
    ("min_ttc_front", np.float64, 0), ("min_ttc_rear", np.float64, 0), ("min_thw", np.float64, 0),
    ("min_ttc_front_tick", np.int64, 0), ("time_hist", np.int32, "hist"),
]


class RolloutSurrogate(C.Structure):
    _fields_ = [(n, _dp) for n, _, _ in SSM_FIELDS]


def rec_mask(triggers) -> int:
    """Recorder trigger mask from an int or an iterable of names of REC_NAMES."""
    if isinstance(triggers, (int, np.integer)):
        return int(triggers)
    mask = 0
    for name in triggers:
        if name not in REC_NAMES:
            raise ValueError(f"unknown recorder trigger {name!r}; expected one of {REC_NAMES}")
        mask |= 1 << REC_NAMES.index(name)
    return mask


def default_config() -> Config:
    """The literals of reference src/main.cpp:30,39-49 (also what
    pp_config_default writes; tests check the two agree)."""
    return Config(5.0, 4.0, 8.0, 22.2, 4.5, 2.0, 10.0, 0.5, 0, 0)


def _inner(kind, max_cars):
    return {0: (), "prev": (PREV_KEEP,), "path": (PATH_LEN,), "cars": (max_cars,)}[kind]


class FrameBatch:
    """N frames in host memory, struct of arrays (numpy), layout of pp_frames."""

    def __init__(self, n: int, max_cars: int = 12):
        self.n = int(n)
        self.max_cars = int(max_cars)
        for name, dt, kind in FRAME_FIELDS:
            setattr(self, name, np.zeros((self.n,) + _inner(kind, self.max_cars), dtype=dt))
        self.target_lane_in[:] = 1

    def arrays(self):
        return {name: getattr(self, name) for name, _, _ in FRAME_FIELDS}

    def struct(self) -> Frames:
        s = Frames()
        for name, dt, _ in FRAME_FIELDS:
            a = getattr(self, name)
            assert a.dtype == dt and a.flags["C_CONTIGUOUS"], name
            setattr(s, name, a.ctypes.data)
        s.max_cars = self.max_cars
        if getattr(self, "car_frozen_lane", None) is not None:  # optional: held-over cars
            for name, dt in FROZEN_FIELDS:
                a = getattr(self, name)
                assert a.dtype == dt and a.flags["C_CONTIGUOUS"] and a.shape == (self.n, self.max_cars), name
                setattr(s, name, a.ctypes.data)
        return s

    def add_frozen(self):
        """Allocate the optional held-over-car arrays (no slot frozen)."""
        for name, dt in FROZEN_FIELDS:
            setattr(self, name, np.zeros((self.n, self.max_cars), dtype=dt))
        self.car_frozen_lane[:] = -1
        return self

    def slice(self, lo: int, hi: int) -> "FrameBatch":
        out = FrameBatch.__new__(FrameBatch)
        out.n = hi - lo
        out.max_cars = self.max_cars
        for name, _, _ in FRAME_FIELDS:
            setattr(out, name, np.ascontiguousarray(getattr(self, name)[lo:hi]))
        return out

    @staticmethod
    def concat(batches) -> "FrameBatch":
        out = FrameBatch.__new__(FrameBatch)
        out.n = sum(b.n for b in batches)
        out.max_cars = batches[0].max_cars
        for name, _, _ in FRAME_FIELDS:
            setattr(out, name, np.ascontiguousarray(
                np.concatenate([getattr(b, name) for b in batches], axis=0)))
        return out

    def bytes_per_frame(self) -> int:
        return sum(a.itemsize * int(np.prod(a.shape[1:], dtype=np.int64))
                   for a in self.arrays().values())


class PlanBatch:
    """N plans in host memory, layout of pp_plans.  `groups` selects which
    optional output groups are allocated (others are passed as NULL)."""

    def __init__(self, n: int, max_cars: int = 12, diag: bool = True, cars: bool = True):
        self.n = int(n)
        self.max_cars = int(max_cars)
        self.fields = list(PLAN_CORE) + (PLAN_DIAG if diag else []) + (PLAN_CARS if cars else [])
        for name, dt, kind in PLAN_FIELDS:
            if name in self.fields:
                a = np.zeros((self.n,) + _inner(kind, self.max_cars), dtype=dt)
                if kind == "path":
                    a[:] = np.nan  # rows beyond n_points are left untouched by every implementation
                setattr(self, name, a)
            else:
                setattr(self, name, None)

    def arrays(self):
        return {name: getattr(self, name) for name in self.fields}

    def struct(self) -> Plans:
        s = Plans()
        for name, dt, _ in PLAN_FIELDS:
            a = getattr(self, name)
            setattr(s, name, None if a is None else a.ctypes.data)
        return s

    def bytes_per_frame(self) -> int:
        return sum(a.itemsize * int(np.prod(a.shape[1:], dtype=np.int64))
                   for a in self.arrays().values())
