"""Test-side binding of tests/incident_oracle.c (TEST INFRASTRUCTURE): the CPU restatement of
the rollouts' incident monitor, built on oracle/pp_oracle.c.  The library is compiled on first
use into a temporary directory (the tree may be read-only), with the oracle's flags."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import checkers

abi = checkers.abi
HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "incident_oracle.c")
_lib = None


def _load():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="pp_incident_oracle_"), "libppincident.so")
        cc = os.environ.get("CC", "gcc")
        subprocess.run([cc, "-O2", "-ffp-contract=off", "-fPIC", "-std=gnu99", "-shared", "-o", out,
                        SRC, "-lm", "-lpthread"], check=True, capture_output=True)
        _lib = C.CDLL(out)
        _lib.ppo_map_create.restype = C.c_void_p
        _lib.ppo_map_create_from_csv.restype = C.c_void_p
    return _lib


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
        self.rec = {name: np.zeros((n, abi.INC_KINDS) if kind else (n,), dtype=dt)
                    for name, dt, kind in abi.INC_FIELDS}
        self.struct = _MonitorStruct(self.ring.ctypes.data, self.pts.ctypes.data,
                                     self.active.ctypes.data, self.off_pts.ctypes.data,
                                     abi.RolloutIncidents(*[a.ctypes.data for a in self.rec.values()]))


class IncidentOracle:
    """The monitor on the highway map (default) or on a map made of the given waypoints."""

    def __init__(self, points=None):
        self.lib = _load()
        if points is None:
            self.map = C.c_void_p(self.lib.ppo_map_create_from_csv(checkers.MAP_CSV.encode()))
        else:
            wx = np.ascontiguousarray(points[0], dtype=np.float64)
            wy = np.ascontiguousarray(points[1], dtype=np.float64)
            self.map = C.c_void_p(self.lib.ppo_map_create(C.c_void_p(wx.ctypes.data),
                                                          C.c_void_p(wy.ctypes.data), C.c_int(len(wx))))
        assert self.map.value, "map creation failed"

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
