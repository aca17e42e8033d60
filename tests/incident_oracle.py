"""Test-side binding of tests/incident_oracle.c (TEST INFRASTRUCTURE): the CPU restatement of
the rollouts' incident monitor, built on oracle/pp_oracle.c
(compiled by sim_oracle.load)."""
from __future__ import annotations

import ctypes as C

import numpy as np

import checkers
import sim_oracle

abi = checkers.abi


class _MonitorStruct(C.Structure):
    """ppo_mon_state of tests/incident_oracle.c."""
    _fields_ = [("ring", C.c_void_p), ("pts", C.c_void_p), ("active", C.c_void_p),
                ("off_pts", C.c_void_p), ("rec", abi.RolloutIncidents)]


class MonitorState:
    """Caller-owned monitor state; `rec` holds the record arrays in the layout
    Rollouts.incidents() returns."""

    def __init__(self, n: int):
        self.n = n
        self.ring = np.zeros((n, abi.INC_HISTORY, 2))
        self.pts = np.zeros(n, np.int64)
        self.active = np.zeros(n, np.uint32)
        self.off_pts = np.zeros(n, np.int32)
        self.rec, rec = abi.host_record(abi.INC_FIELDS, abi.RolloutIncidents, n)
        self.struct = _MonitorStruct(self.ring.ctypes.data, self.pts.ctypes.data,
                                     self.active.ctypes.data, self.off_pts.ctypes.data, rec)


class IncidentOracle:
    """The monitor on the highway map (default) or on a map made of the given waypoints."""

    def __init__(self, points=None):
        self.lib = sim_oracle.load("incident")
        self.map = sim_oracle.make_map(self.lib, points)

    def init(self, ego_x, ego_y) -> MonitorState:
        """A fresh monitor state for len(ego_x) rollouts starting at (ego_x, ego_y)."""
        ms = MonitorState(len(ego_x))
        ex = np.ascontiguousarray(ego_x, dtype=np.float64)
        ey = np.ascontiguousarray(ego_y, dtype=np.float64)
        self.lib.ppo_sim_monitor_init(C.byref(ms.struct), C.c_int64(ms.n), C.c_void_p(ex.ctypes.data),
                                      C.c_void_p(ey.ctypes.data))
        return ms

    def step(self, ms, n_cars, consume_k, frames, plans, before, after):
        """Step `ms` by one tick: the tick's frames and plans, the car states before and after it
        (RolloutStateHost-like objects)."""
        fs, ps = frames.struct(), plans.struct()
        sb, sa = before.struct(), after.struct()
        self.lib.ppo_sim_monitor(self.map, C.byref(ms.struct), C.c_int64(ms.n), C.c_int32(n_cars),
                                 C.c_int32(consume_k), C.byref(fs), C.byref(ps), C.byref(sb),
                                 C.byref(sa))
