"""The flight recorder of the rollouts on the GPU (include/pp.h, pp_rollouts_set_recorder).

The recorded windows are the frames of the last ticks bit for bit; a rollout freezes at its first
incident or non-finite distance; the recorder changes nothing else the rollouts compute; the
windows do not depend on stream groups, graph replay, lean plans, run splitting or sharding; a
replanned window closes the loop bit for bit on the device and within tolerance on the CPU; the
C++ façade reads the same windows as the Python binding.
"""
import mmap
import os
import subprocess

import numpy as np
import pytest

import checkers
import recorder_replay
from test_rollouts import STATE_FIELDS

abi = checkers.abi
INC = abi.INC
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALL_BUT_REAR = [k for k in abi.INC_NAMES if k != "collision_rear"]
FRAME_KEYS = [name for name, _, _ in abi.FRAME_FIELDS]


def _rows(fb, idx):
    return {k: getattr(fb, k)[idx] for k in FRAME_KEYS}


@pytest.mark.gpu
@pytest.mark.parametrize("n,c", [(160, 12), (80, 64)])
@pytest.mark.parametrize("k_first", [1, 3])
def test_recording_is_the_frames_of_the_last_ticks(pp, n, c, k_first):
    w = 7
    ro = pp.Rollouts(pp.Map(), n, c, seed=5, first=300)
    ro.set_recorder(w, 0)
    ks = [k_first] * 5 + [4 - k_first] * 6  # consume_k changes between runs
    history = []
    for t, k in enumerate(ks):
        ro.run(1, k)
        history.append(ro.last()[0])
        rec = ro.recording()
        assert (rec["trigger_tick"] == -1).all() and (rec["trigger_bits"] == 0).all()
        filled = min(t + 1, w)
        for j in range(w):
            rows = np.arange(n) * w + j
            got = _rows(rec["frames"], rows)
            if j < filled:
                tt = t + 1 - filled + j
                assert (rec["tick"][:, j] == tt).all() and (rec["consume_k"][:, j] == ks[tt]).all()
                want = _rows(history[tt], np.arange(n))
                for key in FRAME_KEYS:
                    assert np.array_equal(got[key], want[key]), (t, j, key)
            else:
                assert (rec["tick"][:, j] == -1).all() and (rec["consume_k"][:, j] == 0).all()
                for key in FRAME_KEYS:
                    assert not got[key].any(), (t, j, key)
    # a subset, in any order and with repeats, reads the same rows
    pick = np.array([n - 1, 0, 3, 3])
    sub = ro.recording(pick)
    full = ro.recording()
    assert np.array_equal(sub["tick"], full["tick"][pick])
    rows = (pick[:, None] * w + np.arange(w)).reshape(-1)
    for key in FRAME_KEYS:
        assert np.array_equal(getattr(sub["frames"], key), getattr(full["frames"], key)[rows]), key


@pytest.mark.gpu
def test_recording_of_a_large_index_array_above_4_gb(pp):
    """The index array's address crosses the ABI whole: an anonymous mapping puts the array above
    4 GB, where an address passed as a 32-bit int would be cut."""
    n, w = 70000, 2
    ro = pp.Rollouts(pp.Map(), n, 1, seed=3, lean=True)
    ro.set_recorder(w, 0)
    ro.run(3, 1)
    buf = mmap.mmap(-1, n * 8)
    rows = np.frombuffer(buf, dtype=np.int64)
    rows[:] = np.arange(n)[::-1]
    assert rows.ctypes.data >= 1 << 32
    got, full = ro.recording(rows), ro.recording()
    assert np.array_equal(got["tick"], full["tick"][::-1])
    order = (np.arange(n)[::-1, None] * w + np.arange(w)).reshape(-1)
    for key in FRAME_KEYS:
        assert np.array_equal(getattr(got["frames"], key), getattr(full["frames"], key)[order]), key


def _fast_job(pp, triggers, w=16, ticks=400, n=1024):
    cfg = pp.default_config()
    cfg.max_speed = 25.0  # over-speed fires in most rollouts (test_incidents_fire_through_the_planner)
    ro = pp.Rollouts(pp.Map(), n, 12, seed=31, lean=True)
    ro.set_recorder(w, triggers)
    history = []
    for _ in range(ticks // 50):
        ro.run(50, 1, cfg=cfg)
        history.append(ro.recorder_triggers())
    return ro, history


@pytest.mark.gpu
def test_freezes_at_the_first_incident(pp):
    w, ticks = 16, 400
    ro, history = _fast_job(pp, ALL_BUT_REAR, w, ticks)
    inc, trig = ro.incidents(), ro.recorder_triggers()
    assert np.array_equal(trig["trigger_tick"], inc["first_tick"])
    frozen = trig["trigger_tick"] >= 0
    assert frozen.mean() > 0.5
    assert ((trig["trigger_bits"][frozen] >> inc["first_kind"][frozen]) & 1).all()
    assert (trig["trigger_bits"][~frozen] == 0).all()
    assert (trig["trigger_bits"] & (1 << INC["collision_rear"]) == 0).all()
    # once frozen, a rollout's trigger never moves
    for h in history:
        was = h["trigger_tick"] >= 0
        assert np.array_equal(h["trigger_tick"][was], trig["trigger_tick"][was])
    rec = ro.recording()
    end = np.where(frozen, trig["trigger_tick"], ticks - 1)
    filled = np.minimum(end + 1, w)
    for i in range(ro.n):
        want = np.where(np.arange(w) < filled[i], end[i] - filled[i] + 1 + np.arange(w), -1)
        assert np.array_equal(rec["tick"][i], want), i
    # the window's last frame is the trigger tick's frame: replay a fresh run up to that tick
    i = int(np.flatnonzero(frozen & (trig["trigger_tick"] > 0))[0])
    t = int(trig["trigger_tick"][i])
    cfg = pp.default_config()
    cfg.max_speed = 25.0
    again = pp.Rollouts(pp.Map(), 1024, 12, seed=31, lean=True)
    again.run(t, 1, cfg=cfg)
    again.run(1, 1, cfg=cfg)
    last = _rows(again.last()[0], [i])
    got = _rows(rec["frames"], [i * w + filled[i] - 1])
    for key in FRAME_KEYS:
        assert np.array_equal(got[key], last[key]), key
    # a single-kind mask: only that kind freezes
    ro2, _ = _fast_job(pp, ["off_road"], w, ticks)
    inc2, trig2 = ro2.incidents(), ro2.recorder_triggers()
    assert np.array_equal(inc2["first_tick"], inc["first_tick"])  # the recorder is an observer
    hit = trig2["trigger_tick"] >= 0
    assert (trig2["trigger_bits"][hit] == 1 << INC["off_road"]).all()
    assert (inc2["count"][hit, INC["off_road"]] > 0).all()
    over_speed_only = (inc2["count"][:, INC["over_speed"]] > 0) & (inc2["count"][:, INC["off_road"]] == 0)
    assert over_speed_only.any() and not hit[over_speed_only].any()


# Rollout 169 of profiles/rollout_recorder.py's 64-car IDM job (seed 2026, consume_k 1) is the
# first whose distance turns non-finite, after tick 110 (profiles/rollout_recorder_c64.jsonl).
# Sharding does not change a rollout, so a small job that starts at it reproduces it.
NONFINITE_ROLLOUT, NONFINITE_TICK = 169, 110


@pytest.mark.gpu
def test_freezes_at_a_nonfinite_distance(pp):
    ro = pp.Rollouts(pp.Map(), 8, 64, seed=2026, first=NONFINITE_ROLLOUT, lean=True)
    ro.set_traffic("idm")
    ro.set_recorder(4, ["nonfinite"])
    ro.run(NONFINITE_TICK, 1)
    assert np.isfinite(ro.incidents()["distance_m"][0])
    assert ro.recorder_triggers()["trigger_tick"][0] == -1
    ro.run(1, 1)
    assert not np.isfinite(ro.incidents()["distance_m"][0])
    ro.run(5, 1)
    trig = ro.recorder_triggers()
    assert trig["trigger_tick"][0] == NONFINITE_TICK
    assert trig["trigger_bits"][0] == 1 << abi.REC_NONFINITE
    assert ro.recording([0])["tick"][0].tolist() == list(range(NONFINITE_TICK - 3, NONFINITE_TICK + 1))


def _observed_job(pp, traffic, recorder, c=12, n=4096, ticks=60, k=2):
    ro = pp.Rollouts(pp.Map(), n, c, seed=19)
    ro.set_traffic(traffic)
    if recorder:
        ro.set_recorder(*recorder)
    ro.run(ticks // 2, k)
    ro.run(ticks - ticks // 2, 1)
    st = ro.state()
    out = {f: getattr(st, f) for f in STATE_FIELDS}
    out.update({"incidents." + key: v for key, v in ro.incidents().items()})
    if traffic == "idm":
        out.update({"traffic." + key: v for key, v in ro.traffic().items()})
    fb, pb = ro.last()
    out.update({"frames." + key: v for key, v in fb.arrays().items()})
    out.update({"plans." + key: v for key, v in pb.arrays().items()})
    out["stats"] = ro.stats().cpu().numpy()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("traffic", ["constant", "idm"])
def test_recorder_is_an_observer(pp, traffic):
    ref = _observed_job(pp, traffic, None)
    for rec in ((1, ALL_BUT_REAR), (5, ["nonfinite"]), (64, abi.rec_mask(abi.REC_NAMES))):
        got = _observed_job(pp, traffic, rec)
        for key in ref:
            assert np.array_equal(got[key], ref[key], equal_nan=True), (rec, key)


def _recorded(pp, n=8192, groups=None, lean=False, graph=False, runs=(30,), first=0, w=9):
    cfg = pp.default_config()
    cfg.max_speed = 25.0  # so that some rollouts freeze
    ro = pp.Rollouts(pp.Map(), n, 12, seed=23, first=first, lean=lean)
    ro.set_traffic("idm")
    ro.set_recorder(w, ALL_BUT_REAR)
    if groups is not None:
        ro.set_groups(groups)
    if graph:
        os.environ["PP_ROLLOUT_GRAPH"] = "1"
    try:
        for t in runs:
            ro.run(t, 1, cfg=cfg)
    finally:
        os.environ.pop("PP_ROLLOUT_GRAPH", None)
    rec = ro.recording()
    out = {key: rec[key] for key in ("trigger_tick", "trigger_bits", "tick", "consume_k")}
    out.update({"frames." + key: v for key, v in rec["frames"].arrays().items()})
    return out


@pytest.mark.gpu
def test_recording_does_not_depend_on_groups_graph_lean_run_split_or_sharding(pp):
    ref = _recorded(pp, groups=1, runs=(300,))
    assert (ref["trigger_tick"] >= 0).any() and (ref["trigger_tick"] < 0).any()
    variants = {
        "3 groups, graph replay": _recorded(pp, groups=3, graph=True, runs=(300,)),
        "lean": _recorded(pp, groups=1, lean=True, runs=(300,)),
        "runs of 1, 99, 200": _recorded(pp, runs=(1, 99, 200)),
    }
    for name, got in variants.items():
        for key in ref:
            assert np.array_equal(got[key], ref[key]), (name, key)
    half = 4096
    lo, hi = _recorded(pp, half, runs=(300,)), _recorded(pp, half, runs=(300,), first=half)
    w = 9
    for key in ref:
        cut = half * w if key.startswith("frames.") else half
        assert np.array_equal(ref[key][:cut], lo[key]), ("sharding", key)
        assert np.array_equal(ref[key][cut:], hi[key]), ("sharding", key)


@pytest.mark.gpu
@pytest.mark.parametrize("c", [12, 64])
def test_loop_closure_of_a_replanned_window(pp, oracle, c):
    w, n = 24, 64
    ro = pp.Rollouts(pp.Map(), n, c, seed=41)
    ro.set_traffic("idm")
    ro.set_recorder(w, 0)
    ro.run(30, 1)
    ro.run(30, 2)
    rec = ro.recording()
    fb = rec["frames"]
    m = pp.Map()
    df, dp = pp.DeviceFrames(fb), pp.DevicePlans(fb.n, fb.max_cars, diag=True, cars=True)
    pp.plan_batch(m, df, dp)
    dev = dp.to_host()
    ok, applies = recorder_replay.closure(fb, dev, rec["tick"], rec["consume_k"])
    assert applies.all() and ok.all(), np.argwhere(~ok)[:5]
    cpu = oracle.plan(fb, threads=8)
    ok_cpu, _ = recorder_replay.closure(fb, cpu, rec["tick"], rec["consume_k"], 1e-9, 1e-6)
    assert ok_cpu.all(), np.argwhere(~ok_cpu)[:5]
    assert recorder_replay.oracle_agrees(dev, cpu, n, w, rec["tick"] >= 0).all()


@pytest.mark.gpu
def test_recorder_errors(pp):
    ro = pp.Rollouts(pp.Map(), 64, 12)
    with pytest.raises(pp.PPError):
        ro.recording()  # no recorder
    with pytest.raises(pp.PPError):
        ro.recorder_triggers()
    for window, triggers in ((-1, 0), (abi.REC_MAX_WINDOW + 1, 0), (4, 1 << (abi.REC_NONFINITE + 1)),
                             (4, 1 << 31)):
        with pytest.raises(pp.PPError):
            ro.set_recorder(window, triggers)
    with pytest.raises(ValueError):
        ro.set_recorder(4, ["no_such_kind"])
    ro.set_recorder(abi.REC_MAX_WINDOW, 0)
    ro.set_recorder(0, 0)  # off again, before the first tick: allowed
    ro.set_recorder(3, ["nonfinite"])
    ro.run(1, 1)
    with pytest.raises(pp.PPError):
        ro.set_recorder(3, 0)
    for bad in ([64], [-1], [0, 64]):
        with pytest.raises(pp.PPError):
            ro.recording(bad)
    assert ro.recording([])["tick"].shape == (0, 3)
    assert ro.recording([63])["tick"].tolist() == [[0, -1, -1]]


@pytest.mark.gpu
def test_facade_recording_equals_the_binding(pp, tmp_path):
    exe, out = str(tmp_path / "test_recorder"), str(tmp_path / "rec.bin")
    pkg = os.path.join(ROOT, "carnd-path-planning-project_b200")
    cmd = ["g++", "-std=c++11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "test_recorder.cpp"), "-L", pkg, "-lpp_b200",
           "-Wl,-rpath," + pkg, "-o", exe]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    res = subprocess.run([exe, os.path.join(ROOT, "data", "highway_map.csv"), out],
                         capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and "recorder facade ok" in res.stdout, (res.stdout, res.stderr)
    ro = pp.Rollouts(pp.Map(), 300, 12, seed=11, first=5)
    ro.set_traffic("idm")
    ro.set_recorder(7, 0xFD)
    ro.run(5, 1)
    ro.run(9, 3)
    want = ro.recording([0, 17, 299, 17])
    raw = open(out, "rb").read()
    pos = 0
    order = [("trigger_tick", want["trigger_tick"]), ("trigger_bits", want["trigger_bits"]),
             ("tick", want["tick"]), ("consume_k", want["consume_k"])]
    order += [(k, getattr(want["frames"], k)) for k in ("ego_x", "ego_y", "ego_yaw_deg",
              "ego_speed_mph", "prev_x", "prev_y", "car_x", "car_y", "car_vx", "car_vy",
              "prev_n", "target_lane_in", "n_cars", "car_id")]
    for name, a in order:
        got = np.frombuffer(raw, dtype=a.dtype, count=a.size, offset=pos).reshape(a.shape)
        pos += a.nbytes
        assert np.array_equal(got, a), name
    assert pos == len(raw)
