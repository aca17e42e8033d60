"""The incident monitor of the rollouts (include/pp.h, pp_rollout_incidents) on the CPU: the
oracle's restatement driven with scripted points and car states on a straight road, where every
expectation is exact.  The GPU side is checked against this restatement in test_incidents.py."""
import math

import numpy as np
import pytest

import checkers
import incident_oracle

abi = checkers.abi
INC = abi.INC
SEG = 30.0  # waypoint spacing of the straight road
LANE_Y = [-2.0, -6.0, -10.0]  # lane centres: the reference line is y = 0, d grows to the right


@pytest.fixture(scope="module")
def road():
    """The monitor on a straight road along +x (the scenarios stay far from its wrap-around)."""
    n = 800
    return incident_oracle.IncidentOracle(points=(SEG * np.arange(n), np.zeros(n)))


def car_state(pp, cars):
    """RolloutStateHost of one rollout with cars [(lane, x)] on the straight road."""
    st = pp.RolloutStateHost(1, len(cars))
    for j, (lane, x) in enumerate(cars):
        w = int(x // SEG) + 1
        st.car_lane[0, j] = lane
        st.car_wp[0, j] = w
        st.car_ratio[0, j] = (x - SEG * (w - 1)) / SEG
        st.car_speed[0, j] = 20.0
    return st


def drive(pp, ck, xs, ys, k=1, cars=None):
    """Drive one rollout through the points D_0 = (xs[0], ys[0]), D_1, ... k per tick; cars[t] =
    [(lane, x)] at the start of tick t (len(cars) = ticks + 1).  The record after every tick."""
    xs, ys = np.asarray(xs, float), np.asarray(ys, float)
    ticks = (len(xs) - 1) // k
    nc = len(cars[0]) if cars else 0
    ms = ck.init(xs[:1], ys[:1])
    out = []
    for t in range(ticks):
        fb = abi.FrameBatch(1, max(nc, 1))
        fb.ego_x[0], fb.ego_y[0] = xs[t * k], ys[t * k]
        pb = abi.PlanBatch(1, max(nc, 1), diag=False, cars=False)
        pb.n_points[0] = abi.PATH_LEN
        pb.next_x[0, :k] = xs[t * k + 1:t * k + 1 + k]
        pb.next_y[0, :k] = ys[t * k + 1:t * k + 1 + k]
        pb.ref_wp[0] = int(xs[t * k + k] // SEG) + 1
        before = car_state(pp, cars[t] if cars else [])
        after = car_state(pp, cars[t + 1] if cars else [])
        before.tick = after.tick = t
        ck.step(ms, nc, k, fb, pb, before, after)
        out.append({key: v[0].copy() for key, v in ms.rec.items()})
    return out


def cruise(v, n, x0=600.0, lane=1, offset=0.0):
    """n steps at constant speed v along a lane centre (+ offset to the right)."""
    xs = x0 + v * 0.02 * np.arange(n + 1)
    return xs, np.full(n + 1, LANE_Y[lane] - offset)


def from_speeds(speeds, x0=600.0, lane=1):
    """Points whose step i moves speeds[i] * 0.02 along the lane centre."""
    xs = x0 + np.concatenate([[0.0], np.cumsum(np.asarray(speeds) * 0.02)])
    return xs, np.full(len(xs), LANE_Y[lane])


def counts(rec):
    return {name: int(rec["count"][i]) for name, i in INC.items()}


def test_straight_drive_is_clean(pp, road):
    xs, ys = cruise(20.0, 300)
    recs = drive(pp, road, xs, ys)
    last = recs[-1]
    assert sum(counts(last).values()) == 0
    assert last["first_tick"] == -1 and last["first_kind"] == -1
    want = 0.0
    for i in range(1, len(xs)):  # the same additions in the same order
        want += math.sqrt((xs[i] - xs[i - 1]) ** 2 + (ys[i] - ys[i - 1]) ** 2)
    assert last["distance_m"] == want == last["clean_m"] == last["best_clean_m"]
    assert abs(last["max_speed"] - 20.0) < 1e-9 and last["max_acc"] < 1e-6 and last["max_jerk"] < 1e-6


def test_over_speed_counts_once_at_point_10(pp, road):
    xs, ys = cruise(23.0, 300)
    recs = drive(pp, road, xs, ys)
    assert counts(recs[8])["over_speed"] == 0
    assert counts(recs[9])["over_speed"] == 1  # tick 9 drives point 10, the first defined V
    assert recs[9]["first_tick"] == 9 and recs[9]["first_kind"] == INC["over_speed"]
    assert recs[9]["clean_m"] == 0
    assert all(counts(r)["over_speed"] == 1 for r in recs[9:])
    assert sum(counts(recs[-1]).values()) == 1


def test_velocity_step_is_one_over_acceleration(pp, road):
    # a step of 2.4 m/s between two points: |A| = 2.4 / 0.2 = 12 over one window
    speeds = [15.0] * 150 + [17.4] * 150
    xs, ys = from_speeds(speeds)
    last = drive(pp, road, xs, ys)[-1]
    assert counts(last)["over_acc"] == 1
    assert abs(last["max_acc"] - 12.0) < 1e-6
    assert counts(last)["over_speed"] == 0


def test_acceleration_ramp_is_not_jerk_but_jerk_ramp_is(pp, road):
    # 5 m/s^2 from a 10 m/s cruise up to 22 m/s: within every limit thanks to the 1 s window
    speeds = [10.0] * 100 + [10.0 + 0.1 * i for i in range(1, 121)] + [22.0] * 100
    last = drive(pp, road, *from_speeds(speeds))[-1]
    assert sum(counts(last).values()) == 0
    assert abs(last["max_acc"] - 5.0) < 1e-6 and last["max_jerk"] <= 5.0 + 1e-6
    # a jerk of 15 m/s^3 from a 5 m/s cruise (acceleration 0.3 m/s^2 more every point)
    speeds, v, a = [5.0] * 100, 5.0, 0.0
    for _ in range(70):
        a += 15.0 * 0.02
        v += a * 0.02
        speeds.append(v)
    last = drive(pp, road, *from_speeds(speeds))[-1]
    assert counts(last)["over_jerk"] == 1 and last["max_jerk"] > 10.0


@pytest.mark.parametrize("ticks,want", [(149, 0), (151, 1)])
def test_out_of_lane_after_three_seconds(pp, road, ticks, want):
    xs, ys = cruise(20.0, ticks, offset=1.5)
    recs = drive(pp, road, xs, ys)
    c = counts(recs[-1])
    assert c["out_of_lane"] == want and c["off_road"] == 0 and sum(c.values()) == want
    if want:
        assert recs[149]["first_tick"] == -1 and recs[149]["clean_m"] > 59.0
        assert recs[150]["first_tick"] == 150 and recs[150]["first_kind"] == INC["out_of_lane"]
        assert recs[150]["clean_m"] == 0 and recs[150]["best_clean_m"] == recs[150]["distance_m"]


def test_out_of_lane_count_grows_by_k(pp, road):
    xs, ys = cruise(20.0, 153, offset=1.5)  # k = 3: 51 ticks, 153 points off centre
    recs = drive(pp, road, xs, ys, k=3)
    assert counts(recs[49])["out_of_lane"] == 0  # 150 points
    assert counts(recs[50])["out_of_lane"] == 1 and recs[50]["first_tick"] == 50


def test_off_road(pp, road):
    xs, ys = cruise(20.0, 20)
    ys[:] = -0.5  # d = 0.5
    recs = drive(pp, road, xs, ys)
    assert counts(recs[0])["off_road"] == 1 and recs[0]["first_tick"] == 0
    assert counts(recs[-1])["off_road"] == 1
    assert recs[0]["first_kind"] == INC["off_road"]


def test_collisions(pp, road):
    n, v = 200, 20.0
    xs, ys = cruise(v, n)
    ego = xs
    # a car placed on top of the ego at tick 0, driving along with it: never counted
    cars = [[(1, ego[t])] for t in range(n + 1)]
    last = drive(pp, road, xs, ys, cars=cars)[-1]
    assert sum(counts(last).values()) == 0
    # a faster car closing from behind: one rear collision, clean_m not reset
    cars = [[(1, ego[0] - 20.0 + 25.0 * 0.02 * t)] for t in range(n + 1)]
    recs = drive(pp, road, xs, ys, cars=cars)
    c = counts(recs[-1])
    assert c["collision_rear"] == 1 and sum(c.values()) == 1
    assert recs[-1]["first_tick"] == -1 and recs[-1]["clean_m"] == recs[-1]["distance_m"]
    # the ego closing on a slower car ahead: one front collision, clean_m reset
    cars = [[(1, ego[0] + 20.0 + 15.0 * 0.02 * t)] for t in range(n + 1)]
    recs = drive(pp, road, xs, ys, cars=cars)
    c = counts(recs[-1])
    assert c["collision_front"] == 1 and sum(c.values()) == 1
    t = int(recs[-1]["first_tick"])
    assert recs[-1]["first_kind"] == INC["collision_front"] and recs[t]["clean_m"] == 0
    # gap 20 m closing at 5 m/s: the overlap begins when it is below 4.5 m
    gaps = [ego[0] + 20.0 + 15.0 * 0.02 * s - ego[s] for s in range(n + 1)]
    assert gaps[t] >= 4.5 and gaps[t + 1] < 4.5
    # a car in the next lane passes without a collision
    cars = [[(2, ego[0] - 20.0 + 25.0 * 0.02 * t)] for t in range(n + 1)]
    assert sum(counts(drive(pp, road, xs, ys, cars=cars)[-1]).values()) == 0
