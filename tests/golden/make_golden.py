"""Regenerates the committed golden fixtures (run in the build container, where
/root/reference exists; the GPU box only reads the committed files).

  drawlines_lanes.json   the wpmap / lane0 / lane1 / lane2 arrays the reference's
                         author pasted into DrawLines.ipynb cell 1 (printed with
                         %.4f by reference src/main.cpp:1200-1208) — the only
                         known-answer data for Map::Init in the reference tree.
  frames_c12.npz         768 synthetic frames (12 cars, 30 % steered into rare
  frames_c64.npz         branches) / 96 frames (64 cars): the inputs, and in
  frames_<tag>_out.npz   a file of their own (to keep each file below 1 MB) the
                         outputs of the reference's own code (oracle/_ref/libppref.so).
  units.npz              inputs/outputs of the reference's individual functions.

    python tests/golden/make_golden.py
"""
import json
import os
import re
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from checkers import Checker, load_pkg  # noqa: E402


def drawlines():
    nb = json.load(open("/root/reference/DrawLines.ipynb"))
    src = "".join(nb["cells"][1]["source"])
    out = {}
    for name in ("wpmap", "lane0", "lane1", "lane2"):
        m = re.search(r"^" + name + r"\s*=\s*(\[\[.*?\]\])\s*$", src, re.M | re.S)
        out[name] = json.loads(m.group(1))
        assert len(out[name]) == 181, (name, len(out[name]))
    json.dump(out, open(os.path.join(HERE, "drawlines_lanes.json"), "w"))
    print("drawlines_lanes.json", {k: len(v) for k, v in out.items()})


def frames():
    pp = load_pkg()
    ref = Checker("ref")
    m = pp.Map()
    for tag, n, cars, seed in (("c12", 768, 12, 20261018), ("c64", 96, 64, 20261019)):
        fb = pp.synth_frames(m, n, cars, seed=seed, rare_permille=300)
        plans = ref.plan(fb, want_flags=True)
        blob = {"in_" + k: v for k, v in fb.arrays().items()}
        blob["observable_flags"] = np.uint32(ref.observable_flags)
        np.savez_compressed(os.path.join(HERE, f"frames_{tag}.npz"), **blob)
        np.savez_compressed(os.path.join(HERE, f"frames_{tag}_out.npz"),
                            **{"out_" + k: v for k, v in plans.arrays().items()})
        print(f"frames_{tag}.npz", n, "frames; flag counts",
              {pp.FLAG_NAMES[i]: int(((plans.flags >> i) & 1).sum()) for i in range(pp.NUM_FLAGS)
               if ((plans.flags >> i) & 1).any()})


def units():
    pp = load_pkg()
    ref = Checker("ref")
    m = pp.Map()
    tab = m.table()
    rng = np.random.default_rng(7)
    n = 512
    blob = {}
    # distancesq_pt_seg: generic + clamped + (-1 <= rnom < 0) + degenerate
    a = rng.uniform(-50, 50, (n, 2))
    b = a + rng.uniform(-30, 30, (n, 2))
    p = a + rng.uniform(-60, 60, (n, 2))
    b[:8] = a[:8]                                   # degenerate segment
    p[8:16] = a[8:16] - 1e-3 * (b[8:16] - a[8:16])  # rnom slightly negative
    blob["seg_in"] = np.stack([p[:, 0], p[:, 1], a[:, 0], a[:, 1], b[:, 0], b[:, 1]])
    blob["seg_out"] = np.stack(ref.distancesq_pt_seg(*blob["seg_in"]))
    # points around the track
    w = rng.integers(0, m.n, n)
    u = rng.uniform(0, 1, n)
    lane = rng.integers(0, 3, n)
    off = rng.uniform(-3, 3, n)
    A = tab[(w - 1) % m.n]
    B = tab[w]
    px = A[np.arange(n), 2 + 2 * lane] * (1 - u) + B[np.arange(n), 2 + 2 * lane] * u + B[:, 8] * off
    py = A[np.arange(n), 3 + 2 * lane] * (1 - u) + B[np.arange(n), 3 + 2 * lane] * u + B[:, 9] * off
    px[:16] = tab[w[:16], 0]  # exactly on waypoints: the tie rule
    py[:16] = tab[w[:16], 1]
    blob["ref_in"] = np.stack([px, py])
    wp, ratio = ref.init_reference_waypoint(px, py)
    blob["ref_wp"], blob["ref_ratio"] = wp, ratio
    # objects near each reference point
    ox = px + rng.uniform(-250, 250, n)
    oy = py + rng.uniform(-250, 250, n)
    ox[:64] = px[:64] + rng.uniform(-20, 20, 64)
    oy[:64] = py[:64] + rng.uniform(-20, 20, 64)
    ox[-8:] += 3000  # too far: match fails
    vx = rng.uniform(-25, 25, n)
    vy = rng.uniform(-25, 25, n)
    vx[:4] = 0
    vy[:4] = 1e-7  # |v| < EPSILON branch
    blob["lm_in"] = np.stack([px, py, ox, oy, vx, vy])
    lm = ref.lane_matching(px, py, ox, oy, vx, vy)
    for k, v in lm.items():
        blob["lm_" + k] = v
    s = rng.uniform(-120, 160, n)
    s[:4] = 0.0
    blob["lp_s"], blob["lp_lane"] = s, lane.astype(np.int32)
    lx, ly, lwp, ld = ref.get_lane_pos(px, py, s, lane)
    blob["lp_x"], blob["lp_y"], blob["lp_wp"], blob["lp_dist"] = lx, ly, lwp, ld
    # splines: 3..15 knots, 24 query points each incl. both extrapolation sides and exact knots
    for nk in (3, 6, 13, 15):
        kx = np.cumsum(rng.uniform(0.05, 12, (64, nk)), axis=1) - 20
        ky = rng.uniform(-3, 3, (64, nk))
        q = rng.uniform(kx[:, :1] - 5, kx[:, -1:] + 5, (64, 24))
        q[:, 0] = kx[:, 0]
        q[:, 1] = kx[:, -1]
        q[:, 2] = kx[:, nk // 2]
        blob[f"sp{nk}_kx"], blob[f"sp{nk}_ky"], blob[f"sp{nk}_q"] = kx, ky, q
        blob[f"sp{nk}_out"] = ref.spline(kx, ky, q)
    # Udacity starter helpers on the CSV reference line
    csv = np.loadtxt(pp.MAP_CSV)
    mx, my, ms = csv[:, 0].copy(), csv[:, 1].copy(), csv[:, 2].copy()
    th = rng.uniform(-np.pi, np.pi, n)
    blob["hw_xyth"] = np.stack([px, py, th])
    blob["hw_closest"] = ref.closest_waypoint(px, py, mx, my)
    blob["hw_next"] = ref.next_waypoint(px, py, th, mx, my)
    fs, fd = ref.get_frenet(px, py, th, mx, my)
    blob["hw_frenet"] = np.stack([fs, fd])
    ss = rng.uniform(ms[0] + 1e-3, ms[-1], n)
    dd = rng.uniform(-2, 14, n)
    gx, gy = ref.get_xy(ss, dd, ms, mx, my)
    blob["hw_sd"] = np.stack([ss, dd])
    blob["hw_xy"] = np.stack([gx, gy])
    # LaneChangePlanner / LimitSpeed
    nc = 12
    cid = np.tile(np.arange(nc, dtype=np.int32), (n, 1))
    cs = rng.uniform(-80, 260, (n, nc))
    cvs = rng.uniform(10, 28, (n, nc))
    cl = rng.integers(0, 3, (n, nc)).astype(np.int32)
    cs[:32, 1] = cs[:32, 0]  # ties
    cl[:32, 1] = cl[:32, 0]
    el = rng.integers(0, 3, n).astype(np.int32)
    tl = np.clip(el + rng.integers(-1, 2, n), 0, 2).astype(np.int32)
    es = rng.uniform(-1, 1, n)
    evs = rng.uniform(0, 22, n)
    dt0 = np.where(rng.uniform(0, 1, n) < 0.8, 0.2, 0.0)
    blob["lc_cars"] = np.stack([cs, cvs])
    blob["lc_id"], blob["lc_lane"] = cid, cl
    blob["lc_ego"] = np.stack([es, evs, dt0])
    blob["lc_el"], blob["lc_tl"] = el, tl
    blob["lc_out"] = ref.lane_change(cid, cs, cvs, cl, el, tl, es, evs, dt0)
    cvx = rng.uniform(0, 25, n)
    cvy = rng.uniform(-2, 2, n)
    nxs = rng.uniform(0.5, 60, n)
    espd = rng.uniform(0, 22.2, n)
    eacc = rng.uniform(-6, 6, n)
    inl = rng.integers(0, 2, n).astype(np.int32)
    blob["ls_in"] = np.stack([cvx, cvy, nxs, np.zeros(n), espd, eacc])
    blob["ls_inlane"] = inl
    ls = ref.limit_speed(cvx, cvy, nxs, np.zeros(n), espd, eacc, inl)
    for k, v in ls.items():
        blob["ls_" + k] = v
    # TrajectoryBuilder::build on explicit inputs: take real frames for plausible geometry
    fbt = pp.synth_frames(m, 384, 12, seed=424242, rare_permille=200)
    pl = ref.plan(fbt, want_flags=False)
    tl = np.clip(pl.ego_lane + rng.integers(-1, 2, fbt.n), 0, 2).astype(np.int32)
    sc_target = rng.uniform(0.0, 22.2, fbt.n)
    sc_time = rng.uniform(0.3, 4.0, fbt.n)
    blob["tr_prev_n"], blob["tr_prev_x"], blob["tr_prev_y"] = fbt.prev_n, fbt.prev_x, fbt.prev_y
    blob["tr_ego"] = np.stack([fbt.ego_x, fbt.ego_y, fbt.ego_yaw_deg, pl.ego_d, pl.ego_vd,
                               pl.ego_speed, sc_target, sc_time])
    blob["tr_tl"] = tl
    tx, ty, tn, tf = ref.trajectory_build(fbt.prev_n, fbt.prev_x, fbt.prev_y, fbt.ego_x, fbt.ego_y,
                                          fbt.ego_yaw_deg, tl, pl.ego_d, pl.ego_vd, pl.ego_speed,
                                          sc_target, sc_time)
    blob["tr_x"], blob["tr_y"], blob["tr_n"], blob["tr_flags"] = tx, ty, tn, tf
    np.savez_compressed(os.path.join(HERE, "units.npz"), **blob)
    print("units.npz", len(blob), "arrays")


if __name__ == "__main__":
    drawlines()
    frames()
    units()
