"""Loop closure of recorded rollout windows (include/pp.h, pp_rollouts_set_recorder).

A window holds consecutive frames of one rollout.  Replanning frame j gives plan j, and the
simulator built frame j + 1 from it: with k_j = min(consume_k_j, n_points_j) the ego of frame j + 1
sits at plan j's point k_j - 1 (where it was when k_j = 0), prev_n is n_points_j - k_j, prev_x / y
are plan j's points k_j .. k_j + 9 (0 past prev_n), and target_lane_in is plan j's target_lane.
Used by tests/test_recorder.py, tests/test_recorder_cpu.py and profiles/rollout_recorder.py.
"""
from __future__ import annotations

import numpy as np

PATH_LEN, PREV_KEEP = 50, 10


def _same(a, b, rtol, atol):
    if rtol == 0 and atol == 0:
        return (a == b) | (np.isnan(a) & np.isnan(b))
    return (np.abs(a - b) <= atol + rtol * np.abs(b)) | (np.isnan(a) & np.isnan(b))


def closure(frames, plans, tick, consume_k, rtol=0.0, atol=0.0):
    """frames / plans: m * W frames of m windows and their plans (FrameBatch / PlanBatch);
    tick, consume_k: [m][W].  Returns (ok, applies), both bool [m][W - 1]: transition j -> j + 1
    closes (points bit for bit, or within rtol / atol; integers exactly), and both slots are filled."""
    m, w = tick.shape
    applies = (tick[:, :-1] >= 0) & (tick[:, 1:] >= 0)
    npts = plans.n_points.reshape(m, w)[:, :-1].astype(np.int64)
    k = np.minimum(consume_k[:, :-1], npts)
    nx = plans.next_x.reshape(m, w, PATH_LEN)[:, :-1]
    ny = plans.next_y.reshape(m, w, PATH_LEN)[:, :-1]
    last = np.clip(k - 1, 0, PATH_LEN - 1)[..., None]
    fx, fy = frames.ego_x.reshape(m, w), frames.ego_y.reshape(m, w)
    want_x = np.where(k > 0, np.take_along_axis(nx, last, 2)[..., 0], fx[:, :-1])
    want_y = np.where(k > 0, np.take_along_axis(ny, last, 2)[..., 0], fy[:, :-1])
    ok = _same(fx[:, 1:], want_x, rtol, atol) & _same(fy[:, 1:], want_y, rtol, atol)
    want_n = npts - k
    ok &= frames.prev_n.reshape(m, w)[:, 1:] == want_n
    idx = np.clip(k[..., None] + np.arange(PREV_KEEP), 0, PATH_LEN - 1)
    have = np.arange(PREV_KEEP) < want_n[..., None]
    for got, src in ((frames.prev_x, nx), (frames.prev_y, ny)):
        want = np.where(have, np.take_along_axis(src, idx, 2), 0.0)
        ok &= _same(got.reshape(m, w, PREV_KEEP)[:, 1:], want, rtol, atol).all(axis=2)
    ok &= frames.target_lane_in.reshape(m, w)[:, 1:] == plans.target_lane.reshape(m, w)[:, :-1]
    return ok & applies, applies


def frame_finite(fb):
    """bool [n]: every floating-point field of the frame is finite."""
    fin = np.ones(fb.n, bool)
    for k in ("ego_x", "ego_y", "ego_yaw_deg", "ego_speed_mph", "prev_x", "prev_y", "car_x", "car_y",
              "car_vx", "car_vy"):
        fin &= np.isfinite(getattr(fb, k).reshape(fb.n, -1)).all(axis=1)
    return fin


INT_FIELDS = ("n_points", "ego_lane", "ref_wp", "target_lane", "flags")


def oracle_agrees(dev, cpu, m, w, filled, ints=INT_FIELDS):
    """bool [m]: over the filled slots of each window the CPU plans equal the device plans
    (the integer fields `ints` exactly, points within 1e-9 relative / 1e-6 m, NaN where NaN)."""
    good = np.ones((m, w), bool)
    for k in ints:
        good &= getattr(dev, k).reshape(m, w) == getattr(cpu, k).reshape(m, w)
    for k in ("next_x", "next_y"):
        a, b = getattr(dev, k).reshape(m, w, PATH_LEN), getattr(cpu, k).reshape(m, w, PATH_LEN)
        good &= _same(a, b, 1e-9, 1e-6).all(axis=2)
    return (good | ~filled).all(axis=1)
