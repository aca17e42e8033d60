"""Test-side binding of tests/surrogate_oracle.c (TEST INFRASTRUCTURE): the CPU restatement of
the rollouts' near-miss measures, built on oracle/pp_oracle.c.  The library is compiled on first
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
SRC = os.path.join(HERE, "surrogate_oracle.c")
_lib = None


def _load():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="pp_surrogate_oracle_"), "libppsurrogate.so")
        cc = os.environ.get("CC", "gcc")
        subprocess.run([cc, "-O2", "-ffp-contract=off", "-fPIC", "-std=gnu99", "-shared", "-o", out,
                        SRC, "-lm", "-lpthread"], check=True, capture_output=True)
        _lib = C.CDLL(out)
        _lib.ppo_map_create.restype = C.c_void_p
        _lib.ppo_map_create_from_csv.restype = C.c_void_p
    return _lib


class SurrogateState:
    """Caller-owned record, in the layout Rollouts.surrogate() returns."""

    def __init__(self, n: int):
        self.n = n
        inner = {0: (), "hist": (abi.SSM_MEASURES, abi.SSM_BINS)}
        self.rec = {name: np.zeros((n,) + inner[kind], dtype=dt) for name, dt, kind in abi.SSM_FIELDS}
        self.struct = abi.RolloutSurrogate(*[a.ctypes.data for a in self.rec.values()])


class SurrogateOracle:
    """The measures on the highway map (default) or on a map made of the given waypoints."""

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

    def init(self, n: int) -> SurrogateState:
        ss = SurrogateState(n)
        self.lib.ppo_sim_surrogate_init(C.byref(ss.struct), C.c_int64(n))
        return ss

    def step(self, ss, n_cars, consume_k, frames, plans, after):
        """Step `ss` by one tick: the tick's frames and plans and the car states after it
        (a RolloutStateHost-like object whose tick counts this tick)."""
        fs, ps, sa = frames.struct(), plans.struct(), after.struct()
        self.lib.ppo_sim_surrogate(self.map, C.byref(ss.struct), C.c_int64(ss.n), C.c_int32(n_cars),
                                   C.c_int32(consume_k), C.byref(fs), C.byref(ps), C.byref(sa))
