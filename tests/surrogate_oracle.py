"""Test-side binding of tests/surrogate_oracle.c (TEST INFRASTRUCTURE): the CPU restatement of
the rollouts' near-miss measures, built on oracle/pp_oracle.c
(compiled by sim_oracle.load)."""
from __future__ import annotations

import ctypes as C

import checkers
import sim_oracle

abi = checkers.abi


class SurrogateState:
    """Caller-owned record, in the layout Rollouts.surrogate() returns."""

    def __init__(self, n: int):
        self.n = n
        self.rec, self.struct = abi.host_record(abi.SSM_FIELDS, abi.RolloutSurrogate, n)


class SurrogateOracle:
    """The measures on the highway map (default) or on a map made of the given waypoints."""

    def __init__(self, points=None):
        self.lib = sim_oracle.load("surrogate")
        self.map = sim_oracle.make_map(self.lib, points)

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
