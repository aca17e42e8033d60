"""Test-side binding of tests/traffic_oracle.c (TEST INFRASTRUCTURE): the CPU restatement of the
rollouts' IDM traffic model, built on oracle/pp_oracle.c
(compiled by sim_oracle.load)."""
from __future__ import annotations

import ctypes as C

import numpy as np

import checkers
import sim_oracle

abi = checkers.abi


class TrafficState:
    """Caller-owned IDM state, in the layout Rollouts.traffic() returns."""

    def __init__(self, n: int, n_cars: int):
        self.n, self.n_cars = n, n_cars
        self.arrays, self.struct = abi.host_record(abi.TRAFFIC_FIELDS, abi.RolloutTraffic, n, n_cars)

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
        self.lib = sim_oracle.load("traffic")
        self.map = sim_oracle.make_map(self.lib, points)
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
