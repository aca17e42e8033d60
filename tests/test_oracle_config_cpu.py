"""The CPU oracle with tunables other than the reference's literals, and with cars held over
from earlier messages (no GPU needed).

Every GPU-vs-oracle comparison with a non-default pp_config or with pp_frames::car_frozen_*
trusts the oracle to use them.  A field that both sides ignore would pass such a comparison,
so each tunable is moved here on its own and the output it must move is checked, in closed
form where the reference's arithmetic gives one.
"""
import ctypes as C

import numpy as np
import pytest

import checkers
from conftest import load_golden_frames, plans_dict

abi = checkers.abi
FLAG = abi.FLAG


def same_plans(a, b, skip=()):
    for k in a.fields:
        if k in skip:
            continue
        assert np.array_equal(getattr(a, k), getattr(b, k), equal_nan=True), k


# ---- the default config through the _cfg entry points ---------------------------------------

@pytest.mark.parametrize("source", ["synth12", "synth64", "c12", "c64"])
def test_cfg_entry_points_with_defaults_are_the_plain_ones(pp, pmap, oracle, source):
    if source.startswith("synth"):
        cars = int(source[5:])
        fb = pp.synth_frames(pmap, 3000 if cars == 12 else 600, cars, seed=cars, rare_permille=150)
    else:
        fb = load_golden_frames(abi, source)[0]
    same_plans(oracle.plan(fb, threads=4), oracle.plan(fb, threads=4, cfg=abi.default_config()))


def test_cfg_units_with_defaults_match_golden(oracle, golden_units):
    g, cfg = golden_units, abi.default_config()
    cs, cvs = g["lc_cars"]
    es, evs, dt0 = g["lc_ego"]
    out = oracle.lane_change(g["lc_id"], cs, cvs, g["lc_lane"], g["lc_el"], g["lc_tl"], es, evs,
                             dt0, cfg=cfg)
    assert np.array_equal(out, g["lc_out"])
    ls = oracle.limit_speed(*g["ls_in"], g["ls_inlane"], cfg=cfg)
    for k, v in ls.items():
        assert np.array_equal(v, g["ls_" + k]), k
    ex, ey, yaw, ed, evd, start, target, time = g["tr_ego"]
    ox, oy, on, _ = oracle.trajectory_build(g["tr_prev_n"], g["tr_prev_x"], g["tr_prev_y"], ex, ey,
                                            yaw, g["tr_tl"], ed, evd, start, target, time, cfg=cfg)
    assert np.array_equal(on, g["tr_n"])
    assert np.array_equal(ox, g["tr_x"], equal_nan=True) and np.array_equal(oy, g["tr_y"], equal_nan=True)


def test_reference_checker_refuses_other_configs():
    ref = checkers.Checker.__new__(checkers.Checker)
    ref.kind, ref.pre, ref.lib = "ref", "ppref_", None
    with pytest.raises(ValueError):
        ref._cfg_call("plan_frames", checkers.config("max25"))
    ref.lib = type("L", (), {"ppref_plan_frames": "plain"})()
    assert ref._cfg_call("plan_frames", abi.default_config()) == ("plain", ())


# ---- sensitivity: one tunable at a time ---------------------------------------------------------

@pytest.mark.parametrize("field,value", [("relaxed_acc", 3.0), ("relaxed_acc", 3.9999999999999996),
                                         ("max_speed", 25.0), ("max_speed", 17.5)])
def test_free_road_speed_controller(pp, pmap, oracle, field, value):
    """No car: SpeedController(ego_speed) untouched (src/main.cpp:493-500): target = max_speed,
    time = |v - max_speed| / relaxed_acc."""
    fb = pp.synth_frames(pmap, 2000, 0, seed=7, rare_permille=100, max_cars=1)
    cfg = checkers.config(**{field: value})
    got = oracle.plan(fb, threads=4, cfg=cfg)
    base = oracle.plan(fb, threads=4)
    assert (got.target_speed == cfg.max_speed).all()
    assert np.array_equal(got.target_time, np.abs(got.ego_speed - cfg.max_speed) / cfg.relaxed_acc)
    assert (got.target_time != base.target_time).mean() > 0.9
    assert (got.next_x != base.next_x).any()  # the trajectory follows the controller


def accelerating_frames(pp, pmap, n=3000):
    """Frames whose last kept step is 0.3-1.7 times the one before: ego_acc up to ~±15 m/s^2."""
    fb = pp.synth_frames(pmap, n, 12, seed=9, rare_permille=0)
    fb.prev_n[:] = 47
    k = np.random.default_rng(9).uniform(0.3, 1.7, n)
    for a in (fb.prev_x, fb.prev_y):
        a[:, 9] = a[:, 8] + k * (a[:, 8] - a[:, 7])
    return fb


@pytest.mark.parametrize("maximum_acc", [4.0, 30.0])
def test_maximum_acc_clamps_ego_acc(pp, pmap, oracle, maximum_acc):
    """:1319-1320: ego_acc = clamp(raw, -maximum_acc, maximum_acc)."""
    fb = accelerating_frames(pp, pmap)
    raw = oracle.plan(fb, threads=4, cfg=checkers.config(maximum_acc=1e300)).ego_acc
    assert np.abs(raw).max() > 10.0 and (np.abs(raw) < 4.0).any()
    got = oracle.plan(fb, threads=4, cfg=checkers.config(maximum_acc=maximum_acc))
    assert np.array_equal(got.ego_acc, np.clip(raw, -maximum_acc, maximum_acc))
    assert np.abs(got.ego_acc).max() <= maximum_acc


def limit_speed_rows(cfg, next_s, ego_speed, car_speed, ego_acc):
    n = len(next_s)
    z = np.zeros(n)
    return dict(car_vx=np.full(n, car_speed), car_vy=z, next_s=next_s, ego_s=z,
                ego_speed=np.full(n, ego_speed), ego_acc=np.full(n, ego_acc),
                in_lane=np.ones(n, np.int32))


@pytest.mark.parametrize("field,value", [("keep_distance", 20.0), ("keep_distance_leeway", 0.0),
                                         ("keep_distance_leeway", 3.0)])
def test_keep_and_adjust_move_with_the_keep_distance(pp, pmap, oracle, field, value):
    """A followed car faster than the ego (no braking): ADJUST when it is closer than
    car_length + keep_distance, else KEEP within keep_distance_leeway more (:1112-1140)."""
    flags = {}
    for cfg in (abi.default_config(), checkers.config(**{field: value})):
        L, kd, lw = cfg.car_length, cfg.keep_distance, cfg.keep_distance_leeway
        next_s = np.linspace(4.0, 40.0, 3601)
        r = oracle.limit_speed(**limit_speed_rows(cfg, next_s, 15.0, 20.0, 0.0), cfg=cfg)
        adjust = (0.0 + L + kd) > next_s
        keep = ~adjust & ((0.0 + L + kd + lw) > next_s)
        assert np.array_equal((r["flags"] & FLAG["ADJUST"]) != 0, adjust)
        assert np.array_equal((r["flags"] & FLAG["KEEP"]) != 0, keep)
        assert not (r["flags"] & (FLAG["BRAKE"] | FLAG["MAXBRAKE"])).any()
        assert np.array_equal(r["ls_time"][keep], np.maximum(1.0, np.abs(20.0 - 15.0) / cfg.relaxed_acc)
                              * np.ones(keep.sum()))
        flags[id(cfg)] = r["flags"]
    a, b = flags.values()
    assert (a != b).sum() >= 10
    if field == "keep_distance_leeway" and value == 0.0:  # whole frames: KEEP cannot fire at all
        fb = pp.synth_frames(pmap, 3000, 12, seed=5, rare_permille=0)
        base = oracle.plan(fb, threads=4, cars=False)
        got = oracle.plan(fb, threads=4, cars=False, cfg=checkers.config(keep_distance_leeway=0.0))
        assert (base.flags & FLAG["KEEP"]).any() and not (got.flags & FLAG["KEEP"]).any()


@pytest.mark.parametrize("value", [0.5, 2.5])
def test_braking_deceleration_while_braking(oracle, value):
    """:1082-1100: with ego_acc < 0 the braking distance uses min_relaxed_acc_while_braking;
    BRAKE / MAXBRAKE fire exactly when it exceeds the gap, target time max_dist / (v - dv/2)."""
    n = 2001
    for ego_acc, moves in ((-1.0, True), (1.0, False)):
        out = {}
        for cfg in (abi.default_config(), checkers.config(min_relaxed_acc_while_braking=value)):
            L, sd = cfg.car_length, cfg.safety_distance
            next_s = L + np.linspace(5.0, 420.0, n)
            r = oracle.limit_speed(**limit_speed_rows(cfg, next_s, 20.0, 10.0, ego_acc), cfg=cfg)
            acc = cfg.min_relaxed_acc_while_braking if ego_acc < 0 else cfg.relaxed_acc
            dv = 20.0 - 10.0
            dt = dv / acc
            dd = 20.0 * dt - dv / 2 * dt
            max_dist = (next_s - 0.0 - L) - sd
            brake = dd > max_dist
            hit = (r["flags"] & (FLAG["BRAKE"] | FLAG["MAXBRAKE"])) != 0
            assert np.array_equal(hit, brake)
            soft = (r["flags"] & FLAG["BRAKE"]) != 0
            assert np.array_equal(r["ls_time"][soft], max_dist[soft] / (20.0 - dv / 2))
            assert np.array_equal(r["ls_speed"][brake], np.full(brake.sum(), 10.0))
            out[len(out)] = r
        differ = (out[0]["flags"] != out[1]["flags"]).sum()
        assert (differ > 50) if moves else (differ == 0), (ego_acc, differ)


def lane_frames(oracle, ego_lane, n, speed_mph=20.0):
    """Cold-start frames with the ego on the centre line of `ego_lane`, heading along the road,
    at n waypoints spread over the track."""
    tab = oracle.map_table()
    fb = abi.FrameBatch(n, 1)
    idx = np.linspace(5, len(tab) - 5, n).astype(int)
    a, b = tab[idx - 1, 2 + 2 * ego_lane:4 + 2 * ego_lane], tab[idx, 2 + 2 * ego_lane:4 + 2 * ego_lane]
    p = a + 0.7 * (b - a)
    fb.ego_x[:], fb.ego_y[:] = p[:, 0], p[:, 1]
    fb.ego_yaw_deg[:] = np.degrees(np.arctan2(b[:, 1] - a[:, 1], b[:, 0] - a[:, 0]))
    fb.ego_speed_mph[:] = speed_mph
    fb.prev_n[:] = 0
    fb.target_lane_in[:] = ego_lane
    return fb


def place_car(oracle, fb, s, lane, speed):
    """Car 0 of every frame at arc length s (array) on `lane`'s centre line relative to the ego,
    moving along the lane at `speed`."""
    n = fb.n
    lanes = np.full(n, lane, np.int32)
    x, y, _, _ = oracle.get_lane_pos(fb.ego_x, fb.ego_y, s, lanes)
    x1, y1, _, _ = oracle.get_lane_pos(fb.ego_x, fb.ego_y, s + 1.0, lanes)
    t = np.hypot(x1 - x, y1 - y)
    fb.n_cars[:] = 1
    fb.car_id[:, 0] = 3
    fb.car_x[:, 0], fb.car_y[:, 0] = x, y
    fb.car_vx[:, 0], fb.car_vy[:, 0] = speed * (x1 - x) / t, speed * (y1 - y) / t


@pytest.mark.parametrize("field,value", [("car_length", 8.0), ("safety_distance", 6.0)])
def test_car_behind_in_the_target_lane_threshold(oracle, field, value):
    """:1402: a car counts as next_car_in_target_lane from s0 >= ego_s - car_length -
    safety_distance on; a stopped car behind the ego in its lane is exactly that car or none."""
    fb = lane_frames(oracle, 1, 600)
    place_car(oracle, fb, -np.linspace(2.0, 16.0, fb.n), 1, 0.0)
    picked = {}
    for cfg in (abi.default_config(), checkers.config(**{field: value})):
        p = oracle.plan(fb, threads=4, cfg=cfg)
        assert (p.car_lane[:, 0] == 1).all() and (p.target_lane == 1).all()
        assert (p.next_car_id == -1).all()
        inside = p.car_s[:, 0] >= p.ego_s - cfg.car_length - cfg.safety_distance
        assert inside.any() and not inside.all()
        assert np.array_equal(p.next_car_in_target_lane == 3, inside)
        assert ((p.next_car_in_target_lane == -1) == ~inside).all()
        picked[len(picked)] = inside
    assert (picked[0] != picked[1]).sum() >= 50


def test_fast_lane_change_drops_the_distance_score(oracle):
    """:455-470: with test_fast_lane_change the distance to the old target lane no longer counts.
    Ego in lane 0 behind a car 95 m ahead at 23 m/s: lane 0 scores 22/22.2 + 0.95 (+ 0.5 for
    staying), the empty lane 1 scores 2 (+ 0.25): the default stays, the fast planner moves."""
    fast = checkers.config(test_fast_lane_change=1)
    # the unit: one problem with exactly those values
    args = ([[3]], [[95.0]], [[23.0]], [[0]], [0], [0], [0.0], [0.0], [0.0])
    assert oracle.lane_change(*args)[0] == 0
    assert oracle.lane_change(*args, cfg=fast)[0] == 1
    # whole frames
    fb = lane_frames(oracle, 0, 200)
    place_car(oracle, fb, np.full(fb.n, 95.0), 0, 23.0)
    base = oracle.plan(fb, threads=4)
    got = oracle.plan(fb, threads=4, cfg=fast)
    assert (base.ego_lane == 0).all() and (got.ego_lane == 0).all()
    assert (base.target_lane == 0).all()
    assert (got.target_lane == 1).all()
    assert (got.next_x != base.next_x).any()


# ---- held-over cars --------------------------------------------------------------------------

@pytest.mark.parametrize("cfg_name", ["default", "tight"])
@pytest.mark.parametrize("cars,n", [(12, 2000), (64, 300)])
def test_cars_frozen_at_their_own_values_change_nothing(pp, pmap, oracle, cfg_name, cars, n):
    """Freeze matched cars at exactly what matching gave them and hide their positions (NaN):
    every output stays bit-identical except car_next_wp of the frozen slots, which is 0."""
    cfg = checkers.config(cfg_name)
    fb = pp.synth_frames(pmap, n, cars, seed=20 + cars, rare_permille=150)
    fb.n_cars[::4] = np.random.default_rng(cars).integers(0, cars + 1, len(fb.n_cars[::4]))
    want = oracle.plan(fb, threads=4, cfg=cfg)
    frozen, pick = checkers.hold_over(fb, want, np.random.default_rng(cars), stale=False)
    assert pick.sum() > 0.2 * (want.car_lane >= 0).sum()
    got = oracle.plan(frozen, threads=4, cfg=cfg)
    same_plans(got, want, skip=("car_next_wp",))
    assert (got.car_next_wp[pick] == 0).all()
    assert np.array_equal(got.car_next_wp[~pick], want.car_next_wp[~pick])
    # without the frozen arrays the hidden cars are dropped, and the plans change
    plain = frozen.slice(0, frozen.n)
    del plain.car_frozen_lane
    lost = oracle.plan(plain, threads=4, cfg=cfg)
    assert (lost.car_lane[pick] == -1).all() and (lost.flags & FLAG["CAR_DROPPED"]).any()
    assert (lost.next_car_id != want.next_car_id).any()


def test_stale_frozen_cars_plan_with_their_frozen_values(pp, pmap, oracle):
    fb = pp.synth_frames(pmap, 3000, 12, seed=33, rare_permille=100)
    base = oracle.plan(fb, threads=4)
    frozen, pick = checkers.hold_over(fb, base, np.random.default_rng(33))
    got = oracle.plan(frozen, threads=4)
    for k in ("lane", "s", "d", "vs", "vd"):
        assert np.array_equal(getattr(got, "car_" + k)[pick], getattr(frozen, "car_frozen_" + k)[pick]), k
    assert (got.car_next_wp[pick] == 0).all()
    live = np.arange(fb.max_cars)[None, :] < fb.n_cars[:, None]
    assert (got.car_lane[live & ~pick] == base.car_lane[live & ~pick]).all()
    # the followed cars are sometimes held-over ones, so LimitSpeed saw their car_vx / car_vy
    rows = np.arange(fb.n)
    for k in ("next_car_id", "next_car_in_target_lane"):
        ids = getattr(got, k)
        has = ids >= 0
        j = np.argmax(fb.car_id == ids[:, None], axis=1)
        assert (has & pick[rows, j]).sum() > 20, k
    assert (got.target_speed != base.target_speed).sum() > 50


def test_frame_batch_slice_keeps_the_frozen_arrays(pp, pmap):
    fb = pp.synth_frames(pmap, 10, 4, seed=1).add_frozen()
    fb.car_frozen_lane[3, 1], fb.car_frozen_s[3, 1] = 2, 17.5
    part = fb.slice(2, 5)
    assert part.car_frozen_lane.shape == (3, 4) and part.car_frozen_lane[1, 1] == 2
    assert part.car_frozen_s[1, 1] == 17.5 and part.car_frozen_lane[0, 0] == -1
    s = part.struct()
    assert s.car_frozen_vd == part.car_frozen_vd.ctypes.data
    assert C.c_void_p(s.car_frozen_lane).value == part.car_frozen_lane.ctypes.data
    assert getattr(pp.synth_frames(pmap, 4, 2, seed=1).slice(0, 2), "car_frozen_lane", None) is None
