"""Test-side binding of tests/restart_oracle.c (TEST INFRASTRUCTURE): the CPU restatement of the
rollouts' episode restarts, built on oracle/pp_oracle.c and the monitor's and the IDM model's
restatements (compiled by sim_oracle.load)."""
from __future__ import annotations

import ctypes as C

import numpy as np

import checkers
import incident_oracle
import sim_oracle
import traffic_oracle

abi = checkers.abi


class _RestartStruct(C.Structure):
    """ppo_rst_state of tests/restart_oracle.c."""
    _fields_ = [("count0", C.c_void_p), ("dist0", C.c_void_p), ("rec", abi.RolloutRestarts)]


class RestartState:
    """Caller-owned restart state; `rec` holds the record arrays in the layout
    Rollouts.restarts() returns."""

    def __init__(self, n: int):
        self.n = n
        self.count0 = np.zeros((n, abi.INC_KINDS), np.int32)
        self.dist0 = np.zeros(n)
        self.rec, rec = abi.host_record(abi.RST_FIELDS, abi.RolloutRestarts, n)
        self.struct = _RestartStruct(self.count0.ctypes.data, self.dist0.ctypes.data, rec)


class RestartOracle:
    """The restarts on the highway map (default) or on a map made of the given waypoints.  The
    monitor and the IDM model are the same library's, so their states can be handed over."""

    def __init__(self, points=None):
        self.lib = sim_oracle.load("restart")
        self.lib.ppo_rst_key.restype = C.c_uint64
        self.map = sim_oracle.make_map(self.lib, points)
        self.n_wp = int(C.cast(self.map, C.POINTER(C.c_int))[0])
        self.cum = np.zeros((3, self.n_wp + 1))
        self.lib.ppo_traffic_cum(self.map, C.c_void_p(self.cum.ctypes.data))
        # the monitor and the traffic model, on this library and map
        self.monitor = incident_oracle.IncidentOracle.__new__(incident_oracle.IncidentOracle)
        self.monitor.lib, self.monitor.map = self.lib, self.map
        self.traffic = traffic_oracle.TrafficOracle.__new__(traffic_oracle.TrafficOracle)
        self.traffic.lib, self.traffic.map = self.lib, self.map
        self.traffic.n_wp, self.traffic.cum = self.n_wp, self.cum

    def key(self, seed: int, rollout: int, episode: int) -> int:
        return int(self.lib.ppo_rst_key(C.c_uint64(seed), C.c_int64(rollout), C.c_int64(episode)))

    def draw(self, pp, seed: int, first: int, n: int, n_cars: int, episodes=None):
        """RolloutStateHost of n rollouts drawn as episode episodes[i] (default 0: create's draw)."""
        st = pp.RolloutStateHost(n, n_cars)
        s = st.struct()
        for i in range(n):
            e = 0 if episodes is None else int(episodes[i])
            self.lib.ppo_rst_draw(self.map, C.c_uint64(self.key(seed, first + i, e)), C.c_int32(n_cars),
                                  C.byref(s), C.c_int64(i))
        return st

    def init(self, n: int) -> RestartState:
        return RestartState(n)

    def step(self, rs, state, ms, ts, n_cars, seed, first, mask):
        """The end of a tick: `state` (RolloutStateHost after the tick), the monitor state `ms` and
        the IDM state `ts` (None under constant traffic) restarted in place where `mask` fired."""
        st = state.struct()
        self.lib.ppo_rst_step(self.map, C.c_void_p(self.cum.ctypes.data), C.byref(st),
                              C.byref(ms.struct), C.byref(ts.struct) if ts is not None else None,
                              C.c_int64(state.n), C.c_int32(n_cars), C.c_uint64(seed),
                              C.c_int64(first), C.c_uint32(abi.rec_mask(mask)), C.byref(rs.struct))
