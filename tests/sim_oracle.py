"""Test-side loading of the CPU restatements of the rollouts' observers (TEST INFRASTRUCTURE):
tests/<name>_oracle.c, each built on oracle/pp_oracle.c.  A library is compiled on first use into
a temporary directory (the tree may be read-only), with the oracle's flags."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import checkers

HERE = os.path.dirname(os.path.abspath(__file__))
_libs = {}


def load(name: str):
    """The compiled tests/<name>_oracle.c."""
    if name not in _libs:
        src = os.path.join(HERE, f"{name}_oracle.c")
        out = os.path.join(tempfile.mkdtemp(prefix=f"pp_{name}_oracle_"), f"libpp{name}.so")
        cc = os.environ.get("CC", "gcc")
        subprocess.run([cc, "-O2", "-ffp-contract=off", "-fPIC", "-std=gnu99", "-shared", "-o", out,
                        src, "-lm", "-lpthread"], check=True, capture_output=True)
        lib = C.CDLL(out)
        lib.ppo_map_create.restype = C.c_void_p
        lib.ppo_map_create_from_csv.restype = C.c_void_p
        _libs[name] = lib
    return _libs[name]


def make_map(lib, points=None) -> C.c_void_p:
    """The highway map (points None) or a map made of the waypoints (xs, ys), in `lib`."""
    if points is None:
        m = C.c_void_p(lib.ppo_map_create_from_csv(checkers.MAP_CSV.encode()))
    else:
        wx = np.ascontiguousarray(points[0], dtype=np.float64)
        wy = np.ascontiguousarray(points[1], dtype=np.float64)
        m = C.c_void_p(lib.ppo_map_create(C.c_void_p(wx.ctypes.data), C.c_void_p(wy.ctypes.data),
                                          C.c_int(len(wx))))
    assert m.value, "map creation failed"
    return m
