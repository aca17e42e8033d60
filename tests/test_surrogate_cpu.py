"""The near-miss measures of the rollouts (include/pp.h, pp_rollouts_set_surrogate) on the CPU:
the restatement in surrogate_oracle.c driven with scripted egos and cars on a straight road, where
every expectation is exact.  The GPU side is checked against this restatement in
test_surrogate.py."""
import math

import numpy as np
import pytest

import checkers
import surrogate_oracle

abi = checkers.abi
SEG = 30.0  # waypoint spacing of the straight road
LANE_Y = [-2.0, -6.0, -10.0]  # lane centres: the reference line is y = 0, d grows to the right
FRONT, REAR, THW = abi.SSM["ttc_front"], abi.SSM["ttc_rear"], abi.SSM["thw"]
MINS = ["min_ttc_front", "min_ttc_rear", "min_thw"]
INF = math.inf


@pytest.fixture(scope="module")
def road():
    """The measures on a straight road along +x (the scenarios stay far from its wrap-around)."""
    n = 800
    return surrogate_oracle.SurrogateOracle(points=(SEG * np.arange(n), np.zeros(n)))


def step(pp, ck, ss, t, ego, pts, cars, consume_k=None):
    """Tick t of one rollout: the ego before the tick at `ego`, the plan's points `pts` (k of them
    driven, k = min(consume_k, len(pts)), consume_k defaulting to len(pts)), cars [(lane, x, v)]
    after the tick."""
    nc = max(len(cars), 1)
    fb = abi.FrameBatch(1, nc)
    fb.ego_x[0], fb.ego_y[0] = ego
    pb = abi.PlanBatch(1, nc, diag=False, cars=False)
    pb.n_points[0] = len(pts)
    for j, (x, y) in enumerate(pts):
        pb.next_x[0, j], pb.next_y[0, j] = x, y
    st = pp.RolloutStateHost(1, len(cars))
    for j, (lane, x, v) in enumerate(cars):
        w = int(x // SEG) + 1
        st.car_lane[0, j], st.car_wp[0, j] = lane, w
        st.car_ratio[0, j] = (x - SEG * (w - 1)) / SEG
        st.car_speed[0, j] = v
    st.tick = t + 1
    ck.step(ss, len(cars), len(pts) if consume_k is None else consume_k, fb, pb, st)
    return {k: v[0].copy() for k, v in ss.rec.items()}


def one_tick(pp, ck, cars, k=1, v_ego=20.0, ego_nan=False):
    """A single tick: the ego drives k points at v_ego along lane 1 and ends at P = (605, y1)."""
    y = LANE_Y[1]
    px = 605.0
    pts = [(px - v_ego * 0.02 * (k - 1 - j), y) for j in range(k)]
    ego = (px - v_ego * 0.02 * k, y) if k else (px, y)
    if ego_nan:
        ego, pts = (math.nan, y), [(math.nan, y)] * k
    ss = ck.init(1)
    rec = step(pp, ck, ss, 0, ego, pts, cars)
    u = (px - ego[0]) * 50.0 / k if k else 0.0
    return rec, u


def hist_only(rec, m, b, weight):
    want = np.zeros((abi.SSM_MEASURES, abi.SSM_BINS), np.int32)
    if b is not None:
        want[m, b] = weight
    return np.array_equal(rec["time_hist"][m], want[m])


def test_stopped_car_ahead(pp, road):
    rec, u = one_tick(pp, road, [(1, 645.0, 0.0)])  # centre 40 m ahead of P
    assert rec["min_ttc_front"] == 35.5 / u and abs(rec["min_ttc_front"] - 35.5 / 20) < 1e-9
    assert rec["min_thw"] == 35.5 / u
    assert rec["min_ttc_rear"] == INF
    assert rec["min_ttc_front_tick"] == 0
    assert hist_only(rec, FRONT, 3, 1) and hist_only(rec, THW, 3, 1) and hist_only(rec, REAR, None, 0)


def test_slower_car_ahead_gives_ttc_and_headway(pp, road):
    rec, u = one_tick(pp, road, [(1, 625.0, 15.0)])  # gap 15.5 m, closing at 5 m/s
    assert rec["min_ttc_front"] == 15.5 / (u - 15.0) and abs(rec["min_ttc_front"] - 3.1) < 1e-9
    assert rec["min_thw"] == 15.5 / u
    assert hist_only(rec, FRONT, 5, 1) and hist_only(rec, THW, 1, 1)  # [3, 4) s and [0.5, 1) s


def test_faster_car_ahead_gives_headway_only(pp, road):
    rec, u = one_tick(pp, road, [(1, 625.0, 30.0)])
    assert rec["min_ttc_front"] == INF and rec["min_ttc_front_tick"] == -1
    assert rec["min_thw"] == 15.5 / u
    assert hist_only(rec, FRONT, None, 0) and hist_only(rec, THW, 1, 1)


def test_car_in_the_next_lane_is_not_in_the_path(pp, road):
    rec, _ = one_tick(pp, road, [(2, 625.0, 0.0), (0, 595.0, 40.0)])
    assert [rec[k] for k in MINS] == [INF, INF, INF]
    assert not rec["time_hist"].any()


def test_faster_car_behind_gives_rear_ttc(pp, road):
    rec, u = one_tick(pp, road, [(1, 585.0, 25.0)])  # 20 m behind: gap 15.5 m, closing at 5 m/s
    assert rec["min_ttc_rear"] == 15.5 / (25.0 - u) and abs(rec["min_ttc_rear"] - 3.1) < 1e-9
    assert rec["min_ttc_front"] == INF and rec["min_thw"] == INF
    assert hist_only(rec, REAR, 5, 1) and hist_only(rec, FRONT, None, 0)
    # a slower car behind: nothing
    rec, _ = one_tick(pp, road, [(1, 585.0, 15.0)])
    assert [rec[k] for k in MINS] == [INF, INF, INF]


def test_overlapping_car_is_no_near_miss(pp, road):
    for dx in (3.0, -3.0, 4.0):
        rec, _ = one_tick(pp, road, [(1, 605.0 + dx, 0.0 if dx > 0 else 40.0)])
        assert [rec[k] for k in MINS] == [INF, INF, INF], dx
        assert not rec["time_hist"].any()


def test_weights_and_ego_velocity_of_k(pp, road):
    # k = 0: U = 0, so a stopped car ahead defines nothing and a car behind closes at its speed
    rec, u = one_tick(pp, road, [(1, 645.0, 0.0), (1, 585.0, 10.0)], k=0)
    assert u == 0.0 and rec["min_ttc_front"] == INF and rec["min_thw"] == INF
    assert rec["min_ttc_rear"] == 15.5 / 10.0
    assert hist_only(rec, REAR, 3, 1)  # weight 1 for a tick without a driven point
    # k = 3: weight 3, U from the third point
    rec, u = one_tick(pp, road, [(1, 645.0, 0.0)], k=3)
    assert u == (605.0 - (605.0 - 20.0 * 0.02 * 3)) * 50.0 / 3
    assert rec["min_ttc_front"] == 35.5 / u
    assert hist_only(rec, FRONT, 3, 3) and hist_only(rec, THW, 3, 3)


def test_a_value_on_an_edge_goes_to_the_upper_bin(pp, road):
    rec, _ = one_tick(pp, road, [(1, 550.5, 25.0)], k=0)  # gap 50 m at 25 m/s: exactly 2 s
    assert rec["min_ttc_rear"] == 2.0
    assert hist_only(rec, REAR, 4, 1)  # [2, 3), not [1.5, 2)
    rec, _ = one_tick(pp, road, [(1, 529.5, 10.0)], k=0)  # gap 71 m at 10 m/s: 7.1 s
    assert hist_only(rec, REAR, 7, 1)
    rec, _ = one_tick(pp, road, [(1, 519.5, 10.0)], k=0)  # gap 81 m: 8.1 s, not counted
    assert rec["min_ttc_rear"] == 8.1 and not rec["time_hist"].any()


def test_nan_ego_defines_nothing(pp, road):
    rec, _ = one_tick(pp, road, [(1, 645.0, 0.0), (1, 585.0, 25.0)], ego_nan=True)
    assert [rec[k] for k in MINS] == [INF, INF, INF] and rec["min_ttc_front_tick"] == -1
    assert not rec["time_hist"].any()


def test_min_tick_moves_only_on_a_strict_decrease(pp, road):
    y = LANE_Y[1]
    ss = road.init(1)
    ego, pts = (604.6, y), [(605.0, y)]
    recs = [step(pp, road, ss, t, ego, pts, [(1, x, 0.0)])
            for t, x in enumerate([645.0, 645.0, 635.0, 635.0, 655.0, 625.0])]
    assert [int(r["min_ttc_front_tick"]) for r in recs] == [0, 0, 2, 2, 2, 5]
    u = (605.0 - 604.6) * 50.0
    assert [float(r["min_ttc_front"]) for r in recs] == [35.5 / u] * 2 + [25.5 / u] * 3 + [15.5 / u]
    # six ticks of weight 1 in the front TTC histogram: 1.78 s x 2 in [1.5, 2), 1.28 s x 2 and
    # 2.78 s in [1, 1.5) and [2, 3), 0.78 s in [0.5, 1)
    assert recs[-1]["time_hist"][FRONT].tolist() == [0, 1, 2, 2, 1, 0, 0, 0]
