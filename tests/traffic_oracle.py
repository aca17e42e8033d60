"""Test-side binding of tests/traffic_oracle.c (TEST INFRASTRUCTURE): the CPU restatement of the
rollouts' IDM traffic model, built on oracle/pp_oracle.c.  The library is compiled on first use
into a temporary directory (the tree may be read-only), with the oracle's flags."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import checkers

abi = checkers.abi
HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "traffic_oracle.c")
_lib = None


def _load():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="pp_traffic_oracle_"), "libpptraffic.so")
        cc = os.environ.get("CC", "gcc")
        subprocess.run([cc, "-O2", "-ffp-contract=off", "-fPIC", "-std=gnu99", "-shared", "-o", out,
                        SRC, "-lm", "-lpthread"], check=True, capture_output=True)
        _lib = C.CDLL(out)
        _lib.ppo_map_create.restype = C.c_void_p
        _lib.ppo_map_create_from_csv.restype = C.c_void_p
    return _lib


class TrafficState:
    """Caller-owned IDM state, in the layout Rollouts.traffic() returns."""

    def __init__(self, n: int, n_cars: int):
        inner = {"cars": (n_cars,), 0: (), "lanes": (3,)}
        self.n, self.n_cars = n, n_cars
        self.arrays = {name: np.zeros((n,) + inner[kind], dtype=dt)
                       for name, dt, kind in abi.TRAFFIC_FIELDS}
        self.struct = abi.RolloutTraffic(*[a.ctypes.data for a in self.arrays.values()])

    def __getitem__(self, name):
        return self.arrays[name]

    def copy(self):
        out = TrafficState(self.n, self.n_cars)
        for k, a in self.arrays.items():
            out.arrays[k][...] = a
        return out


class TrafficOracle:
    """The IDM model on the highway map (default) or on a map made of the given waypoints."""

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
        self.n_wp = int(C.cast(self.map, C.POINTER(C.c_int))[0])
        self.cum = np.zeros((3, self.n_wp + 1))
        self.lib.ppo_traffic_cum(self.map, C.c_void_p(self.cum.ctypes.data))

    def init(self, state) -> TrafficState:
        """The state selecting the model gives: v0 = speed, acc = 0, the ego's initial lane state."""
        ts = TrafficState(state.n, state.n_cars)
        st = state.struct()
        self.lib.ppo_traffic_init(self.map, C.c_void_p(self.cum.ctypes.data), C.byref(st),
                                  C.c_int64(state.n), C.c_int32(state.n_cars), C.byref(ts.struct))
        return ts

    def advance(self, state, ts, seed, first, consume_k, plans):
        """One tick: `state` (a RolloutStateHost with path_x / path_y) and `ts` stepped in place."""
        st = state.struct()
        ps = plans.struct()
        self.lib.ppo_sim_advance_idm(self.map, C.c_void_p(self.cum.ctypes.data), C.byref(st),
                                     C.byref(ts.struct), C.c_int64(state.n), C.c_int32(state.n_cars),
                                     C.c_uint64(seed), C.c_int64(first), C.c_int32(consume_k),
                                     C.byref(ps))
        state.tick = int(st.tick)
